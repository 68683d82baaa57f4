// spx_common.cuh -- shared device/host plumbing of libshiftedprox (sm_100a only).
//
// Arithmetic contract (SURVEY.md Appendix A): IEEE-754 round-to-nearest, no FMA
// contraction (the library is compiled with -fmad=false), no reassociation,
// Julia's min/max/sign semantics.  All helpers here are branch-free selects.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <cstdio>
#include <limits>

#include "../../include/shiftedprox.h"

#ifndef __CUDA_ARCH_LIST__
#define __CUDA_ARCH_LIST__ 1000
#endif

namespace spx {

// ------------------------------------------------------------------ errors --
void set_error(const char* fmt, ...);
int32_t cuda_fail(cudaError_t e, const char* what);

#define SPX_CUDA(call)                                       \
  do {                                                       \
    cudaError_t e__ = (call);                                \
    if (e__ != cudaSuccess) return spx::cuda_fail(e__, #call); \
  } while (0)

#define SPX_REQUIRE(cond, msg)                 \
  do {                                         \
    if (!(cond)) {                             \
      spx::set_error("%s: %s", __func__, msg); \
      return SPX_E_INVALID;                    \
    }                                          \
  } while (0)

// ----------------------------------------------------------------- context --
// Reduction scratch: one (sum, flag) slot per block of the producing kernel,
// folded in fixed order by a single-block kernel -> deterministic for a given n.
struct Partial {
  double s;       // Σ of whatever h accumulates (|v|, v≠0, √|v|, ...)
  double s2;      // second accumulator (Σw² of the L2 trust-region term, ...)
  long long bad;  // infeasibility flag / min index of a failed assertion (max-reduced)
};

constexpr int kMaxPartials = 148 * 32;
constexpr int kMaxScale = 16;  // simultaneous trial scalings of one L1B2 pass

}  // namespace spx

struct spx_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  bool owns_stream = false;
  spx::Partial* d_partials = nullptr;  // kMaxPartials * kMaxScale slots
  spx::Partial* d_result = nullptr;    // kMaxScale slots
  spx::Partial* h_result = nullptr;    // pinned mirror
  void* d_scratch = nullptr;           // histogram / select state
  size_t scratch_bytes = 0;
  // host-buffer pipeline (spx_box_host_*): lazily created
  cudaStream_t pipe_streams[3] = {nullptr, nullptr, nullptr};
  void* pipe_buf = nullptr;
  size_t pipe_bytes = 0;
  // fork / join of side streams 0 and 1 by the group kernels (spx_group.cu): lazily created
  cudaEvent_t pipe_events[3] = {};
  long long launches = 0;
  // multi-GPU (spx_comm.cu): an NCCL communicator bound to this context's device and stream
  void* comm = nullptr;  // ncclComm_t
  int comm_nranks = 1, comm_rank = 0;
  bool reduce_scalars = false;  // every folded reduction is all-reduced on the device before it reaches the host
  double* d_comm = nullptr;     // packed scalars of a multi-slot reduction
  long long collectives = 0;
  // peer-memory exchange (spx_comm_peer_*): every rank's exchange buffer mapped into this process over NVLink;
  // the fold kernel of a reduction then finishes the all-reduce itself (stores into the peers, spin on its own buffer)
  void* peer_own = nullptr;        // this rank's exchange buffer (cudaMalloc, exported by IPC handle)
  void** d_peer_ptrs = nullptr;    // device array [nranks]: every rank's exchange buffer as seen from here
  void* peer_mapped[16] = {};      // host copies of the mapped pointers (closed on destroy)
  int peer_nranks = 0;
  unsigned long long peer_seq = 0;  // all-reduces done so far (the same number on every rank)
  int* d_peer_fail = nullptr;
  // size classes present in the CSR layouts validated on this context (spx_group_validate_offsets): lets the group
  // entry points skip the CTA-per-group launches of an absent class.  A hint only: the warp kernels are told which
  // classes were skipped and take their groups themselves, so a stale entry costs time, never a result.
  struct GroupCensus {
    const void* offs = nullptr;
    long long ngroups = -1, n = -1;
    unsigned classes = 0;  // bit 0: some group of 257..1024 elements, bit 1: of 1025..4096, bit 2: longer ones
  } census[8];
  int census_next = 0;
};

namespace spx {

int32_t ensure_scratch(spx_ctx* ctx, size_t bytes);

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

// ------------------------------------------------------------ Julia Base.* --
// Base.min/max on IEEE floats: NaN-propagating, min(-0.0, 0.0) = -0.0.
template <class R> __host__ __device__ __forceinline__ bool sgnbit(R x);
template <> __host__ __device__ __forceinline__ bool sgnbit<double>(double x) {
#ifdef __CUDA_ARCH__
  return __double2hiint(x) < 0;
#else
  return std::signbit(x);
#endif
}
template <> __host__ __device__ __forceinline__ bool sgnbit<float>(float x) {
#ifdef __CUDA_ARCH__
  return __float_as_int(x) < 0;
#else
  return std::signbit(x);
#endif
}
template <class R> __host__ __device__ __forceinline__ R jl_min(R x, R y) {
  R diff = x - y;
  R arg = sgnbit(diff) ? x : y;
  return (x != x || y != y) ? diff : arg;
}
template <class R> __host__ __device__ __forceinline__ R jl_max(R x, R y) {
  R diff = x - y;
  R arg = sgnbit(diff) ? y : x;
  return (x != x || y != y) ? diff : arg;
}
// Base.sign: sign(±0.0) = ±0.0, sign(NaN) = NaN
template <class R> __host__ __device__ __forceinline__ R jl_sign(R x) {
  return x > R(0) ? R(1) : (x < R(0) ? R(-1) : x);
}
template <class R> __host__ __device__ __forceinline__ R jl_abs(R x) { return x < R(0) ? -x : (x == R(0) ? R(0) : x); }
template <> __host__ __device__ __forceinline__ double jl_abs<double>(double x) { return fabs(x); }
template <> __host__ __device__ __forceinline__ float jl_abs<float>(float x) { return fabsf(x); }

template <class R> struct Eps;
template <> struct Eps<double> {
  static constexpr double value = 2.220446049250313e-16;      // eps(Float64)
  static constexpr double sqrt_value = 1.4901161193847656e-8;  // √eps(Float64)
};
template <> struct Eps<float> {
  static constexpr float value = 1.1920929e-7f;          // eps(Float32)
  static constexpr float sqrt_value = 0.00034526698f;     // √eps(Float32) = Float32(2^-11.5)
};

// ShiftedProximalOperators.jl:203
template <class R> __host__ __device__ __forceinline__ R prox_zero(R q, R l, R u) {
  return jl_min(jl_max(q, l), u);
}
// ShiftedProximalOperators.jl:217-236
template <class R> __host__ __device__ __forceinline__ R iprox_zero(R d, R g, R l, R u) {
  const R eps = Eps<R>::value;
  R r;
  if (d > eps) {
    R argmin_quad = (-g) / d;
    r = jl_min(jl_max(argmin_quad, l), u);
  } else if (d < -eps) {
    R d_2 = d / R(2);
    R val_l = d_2 * (l * l) + g * l;
    R val_u = d_2 * (u * u) + g * u;
    r = (val_l < val_u) ? l : u;
  } else {
    r = (g > R(0)) ? l : ((g < R(0)) ? u : R(0));
  }
  return r;
}

// ------------------------------------------------- 128-bit streaming access --
// Every operand is touched exactly once: bypass L1 allocation on loads, and
// mark stores streaming.  No `.nc`: y may alias q (test/test_allocs.jl:108).
#ifdef __CUDACC__
template <class R, int VEC> struct Pack { R v[VEC]; };

__device__ __forceinline__ void ld_stream(const double* p, Pack<double, 2>& o) {
  asm volatile("ld.global.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(o.v[0]), "=d"(o.v[1]) : "l"(p));
}
__device__ __forceinline__ void ld_stream(const double* p, Pack<double, 1>& o) {
  asm volatile("ld.global.L1::no_allocate.f64 %0, [%1];" : "=d"(o.v[0]) : "l"(p));
}
__device__ __forceinline__ void ld_stream(const float* p, Pack<float, 4>& o) {
  asm volatile("ld.global.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(o.v[0]), "=f"(o.v[1]), "=f"(o.v[2]), "=f"(o.v[3])
               : "l"(p));
}
__device__ __forceinline__ void ld_stream(const float* p, Pack<float, 1>& o) {
  asm volatile("ld.global.L1::no_allocate.f32 %0, [%1];" : "=f"(o.v[0]) : "l"(p));
}
__device__ __forceinline__ void st_stream(double* p, const Pack<double, 2>& o) {
  asm volatile("st.global.cs.v2.f64 [%0], {%1, %2};" ::"l"(p), "d"(o.v[0]), "d"(o.v[1]) : "memory");
}
__device__ __forceinline__ void st_stream(double* p, const Pack<double, 1>& o) {
  asm volatile("st.global.cs.f64 [%0], %1;" ::"l"(p), "d"(o.v[0]) : "memory");
}
__device__ __forceinline__ void st_stream(float* p, const Pack<float, 4>& o) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(o.v[0]), "f"(o.v[1]),
               "f"(o.v[2]), "f"(o.v[3])
               : "memory");
}
__device__ __forceinline__ void st_stream(float* p, const Pack<float, 1>& o) {
  asm volatile("st.global.cs.f32 [%0], %1;" ::"l"(p), "f"(o.v[0]) : "memory");
}

// ------------------------------------------------- asynchronous copies to shared memory --
// Per-thread 16-byte cp.async (LDGSTS), completed by cp.async.wait_group, and 16-byte shared loads.
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void lds16(uint32_t a, Pack<double, 2>& o) {
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(o.v[0]), "=d"(o.v[1]) : "r"(a) : "memory");
}
__device__ __forceinline__ void lds16(uint32_t a, Pack<float, 4>& o) {
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(o.v[0]), "=f"(o.v[1]), "=f"(o.v[2]), "=f"(o.v[3])
               : "r"(a)
               : "memory");
}

// Bulk copies (cp.async.bulk, UBLKCP): one thread moves a contiguous run of 16-byte granules global -> shared, and
// the copy completes on an mbarrier (expect_tx / complete_tx): no LSU instructions, no registers, any thread of the
// CTA may read the run once the barrier's phase flips.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tSPX_MBAR_WAIT:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra SPX_MBAR_DONE;\n\t"
      "bra SPX_MBAR_WAIT;\n\tSPX_MBAR_DONE:\n\t}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// orders the CTA's earlier generic-proxy reads of a buffer before the async-proxy writes of the next bulk copy into it
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// --------------------------------------------------------------- reductions --
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ long long warp_max(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    long long t = __shfl_xor_sync(0xffffffffu, v, o);
    v = t > v ? t : v;
  }
  return v;
}
// Block-wide fold of a Partial; result valid in thread 0.  Fixed order.
template <int THREADS> __device__ __forceinline__ Partial block_fold(Partial p) {
  __shared__ double sh_s[THREADS / 32], sh_s2[THREADS / 32];
  __shared__ long long sh_b[THREADS / 32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  p.s = warp_sum(p.s);
  p.s2 = warp_sum(p.s2);
  p.bad = warp_max(p.bad);
  if (lane == 0) { sh_s[w] = p.s; sh_s2[w] = p.s2; sh_b[w] = p.bad; }
  __syncthreads();
  if (w == 0) {
    Partial t;
    t.s = lane < THREADS / 32 ? sh_s[lane] : 0.0;
    t.s2 = lane < THREADS / 32 ? sh_s2[lane] : 0.0;
    t.bad = lane < THREADS / 32 ? sh_b[lane] : -1;
    t.s = warp_sum(t.s);
    t.s2 = warp_sum(t.s2);
    t.bad = warp_max(t.bad);
    p = t;
  }
  __syncthreads();
  return p;
}
#endif  // __CUDACC__

// `selected` on the device (see spx_sel in the header)
struct DevSel {
  int kind;
  long long start, step, stop;
  const uint32_t* mask;
  __host__ __device__ __forceinline__ bool has(long long i) const {
    if (kind == SPX_SEL_ALL) return true;
    if (kind == SPX_SEL_RANGE) {
      if (i < start || i > stop) return false;
      unsigned long long off = (unsigned long long)(i - start);
      if ((stop >> 32) == 0) return ((unsigned)off % (unsigned)step) == 0u;
      return (off % (unsigned long long)step) == 0ull;
    }
#ifdef __CUDA_ARCH__
    return (__ldg(mask + (i >> 5)) >> (i & 31)) & 1u;
#else
    return (mask[i >> 5] >> (i & 31)) & 1u;
#endif
  }
};

int32_t make_sel(const spx_sel* s, int64_t n, DevSel* out);

// fold `nblocks` partials (slot stride `stride`, `nslot` independent slots) into
// ctx->d_result[slot], copy to the pinned mirror, synchronise
int32_t finalize_partials(spx_ctx* ctx, int nblocks, int nslot, bool bad_is_min);
// the two passes of the solver step around a prox! that is not one streaming pass (spx_step.cu)
template <class R> int32_t step_pre(spx_ctx* ctx, int64_t n, R* q, const R* grad, double nu);
template <class R>
int32_t step_post(spx_ctx* ctx, int64_t n, R* xsy, const R* xk, const R* sj, const R* s, const R* grad, double* out2);
// the finish pass of the ShiftedNormL1B2 step (spx_step.cu, called by the root search of spx_l1b2.cu)
template <class R>
int32_t step_l1b2_finish(spx_ctx* ctx, int64_t n, R* s, R* xsy, const R* xk, const R* sj, const R* grad, const R* mid,
                         R nu, R ls, bool use_scale, R scale, R post, double* v);
// spx_comm.cu: is the context in "scalars are global" mode; all-reduce ctx->d_result[0..nslot) on ctx->stream
bool comm_active(const spx_ctx* ctx);
int32_t comm_neutral_result(spx_ctx* ctx, int nslot);
int32_t comm_allreduce_result(spx_ctx* ctx, int nslot);
int32_t comm_allreduce_raw(spx_ctx* ctx, void* buf, size_t count, int nccl_dtype, int nccl_op);
// ncclDataType_t / ncclRedOp_t values (checked against nccl.h in spx_comm.cu), for callers that do not include nccl.h
constexpr int kNcclInt64 = 4, kNcclUint64 = 5, kNcclFloat64 = 8, kNcclSum = 0, kNcclMax = 2;
// spx_comm.cu: fold + all-reduce over peer memory in ONE kernel (when the exchange buffers are attached)
bool comm_peer_ready(const spx_ctx* ctx);
int32_t comm_fold_allreduce_peer(spx_ctx* ctx, int nblocks, int nslot);
// enqueue only: fold `nblocks` partials at `partials` into *result on `stream`
int32_t enqueue_fold(spx_ctx* ctx, cudaStream_t stream, const Partial* partials, int nblocks, Partial* result);

// internal launchers shared across translation units -------------------------
// op codes of the Box family
enum BoxOp { BOX_L1 = 0, BOX_L0 = 1, BOX_LHALF = 2 };

template <class R>
int32_t launch_box(spx_ctx* ctx, cudaStream_t stream, int op, bool inverse, int64_t n, R* y,
                   const R* xk, const R* sj, const R* qg, const R* d, const R* lvec, R lval,
                   const R* uvec, R uval, DevSel sel, R lambda, R sigma, bool want_psi,
                   Partial* partials, int* nblocks_out, int64_t index_base);

}  // namespace spx
