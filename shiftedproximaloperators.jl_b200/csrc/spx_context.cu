// spx_context.cu -- context, device buffers, state ops (shift!/set_bounds!/ctor
// checks), synthetic-input generator and checksum of libshiftedprox.
#include <cstdarg>
#include <cstring>

#include "spx_elementwise.cuh"

namespace spx {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int32_t cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
  return (int32_t)e;
}

int32_t ensure_scratch(spx_ctx* ctx, size_t bytes) {
  if (ctx->scratch_bytes >= bytes) return SPX_OK;
  if (ctx->d_scratch) {
    SPX_CUDA(cudaStreamSynchronize(ctx->stream));
    SPX_CUDA(cudaFree(ctx->d_scratch));
    ctx->d_scratch = nullptr;
    ctx->scratch_bytes = 0;
  }
  SPX_CUDA(cudaMalloc(&ctx->d_scratch, bytes));
  ctx->scratch_bytes = bytes;
  return SPX_OK;
}

int32_t make_sel(const spx_sel* s, int64_t n, DevSel* out) {
  DevSel d;
  d.kind = SPX_SEL_ALL;
  d.start = 0;
  d.step = 1;
  d.stop = n - 1;
  d.mask = nullptr;
  if (s != nullptr) {
    d.kind = s->kind;
    if (s->kind == SPX_SEL_RANGE) {
      if (s->step <= 0) {
        set_error("spx_sel: RANGE needs step > 0");
        return SPX_E_INVALID;
      }
      d.start = s->start;
      d.step = s->step;
      d.stop = s->stop < n - 1 ? s->stop : n - 1;
      if (d.start == 0 && d.step == 1 && d.stop == n - 1) d.kind = SPX_SEL_ALL;
    } else if (s->kind == SPX_SEL_MASK) {
      if (s->mask == nullptr) {
        set_error("spx_sel: MASK needs a device mask");
        return SPX_E_INVALID;
      }
      d.mask = s->mask;
    } else if (s->kind != SPX_SEL_ALL) {
      set_error("spx_sel: unknown kind %d", (int)s->kind);
      return SPX_E_INVALID;
    }
  }
  *out = d;
  return SPX_OK;
}

// Fold the per-block partials of up to kMaxScale slots; slot k lives at
// partials[k * nblocks .. (k+1) * nblocks).  One block per slot, fixed order.
__global__ void __launch_bounds__(256) fold_kernel(const Partial* __restrict__ partials, int nblocks,
                                                   Partial* __restrict__ result) {
  const Partial* p = partials + (size_t)blockIdx.x * nblocks;
  Partial acc;
  acc.s = 0.0;
  acc.s2 = 0.0;
  acc.bad = -1;
  for (int i = threadIdx.x; i < nblocks; i += 256) {
    Partial t = p[i];
    acc.s += t.s;
    acc.s2 += t.s2;
    acc.bad = t.bad > acc.bad ? t.bad : acc.bad;
  }
  acc = block_fold<256>(acc);
  if (threadIdx.x == 0) result[blockIdx.x] = acc;
}

int32_t enqueue_fold(spx_ctx* ctx, cudaStream_t stream, const Partial* partials, int nblocks, Partial* result) {
  fold_kernel<<<1, 256, 0, stream>>>(partials, nblocks, result);
  ctx->launches++;
  SPX_CUDA(cudaGetLastError());
  return SPX_OK;
}

int32_t finalize_partials(spx_ctx* ctx, int nblocks, int nslot, bool) {
  const bool global = comm_active(ctx);  // sharded vector: the folded slots are all-reduced on the device
  if (nblocks <= 0 && !global) {
    for (int k = 0; k < nslot; ++k) {
      ctx->h_result[k].s = 0.0;
      ctx->h_result[k].s2 = 0.0;
      ctx->h_result[k].bad = -1;
    }
    return SPX_OK;
  }
  if (global && comm_peer_ready(ctx)) {
    // one kernel: fold this rank's partials, store the folded slots into every peer's exchange buffer over NVLink,
    // wait for the peers' slots in our own buffer, sum in rank order (identical bits on every rank)
    int32_t st = comm_fold_allreduce_peer(ctx, nblocks, nslot);
    if (st != SPX_OK) return st;
    SPX_CUDA(cudaMemcpyAsync(ctx->h_result, ctx->d_result, sizeof(Partial) * nslot, cudaMemcpyDeviceToHost, ctx->stream));
    SPX_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < nslot; ++k)
      if (ctx->h_result[k].bad == (1ll << 61)) {
        set_error("peer all-reduce timed out: a rank did not reach the same reduction");
        return SPX_E_INVALID;
      }
    return SPX_OK;
  }
  if (nblocks > 0) {
    fold_kernel<<<nslot, 256, 0, ctx->stream>>>(ctx->d_partials, nblocks, ctx->d_result);
    ctx->launches++;
    SPX_CUDA(cudaGetLastError());
  } else {  // an empty shard still takes part in the collective
    int32_t st = comm_neutral_result(ctx, nslot);
    if (st != SPX_OK) return st;
  }
  if (global) {
    int32_t st = comm_allreduce_result(ctx, nslot);
    if (st != SPX_OK) return st;
  }
  SPX_CUDA(cudaMemcpyAsync(ctx->h_result, ctx->d_result, sizeof(Partial) * nslot, cudaMemcpyDeviceToHost,
                           ctx->stream));
  SPX_CUDA(cudaStreamSynchronize(ctx->stream));
  return SPX_OK;
}

// ------------------------------------------------------------ small kernels --
// strided copy (strides in elements): the gather / scatter between a strided `SubArray` shift and its contiguous shadow
template <class W>
__global__ void __launch_bounds__(256) copy_strided_kernel(long long n, W* __restrict__ dst, long long ds,
                                                           const W* __restrict__ src, long long ss) {
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256)
    dst[i * ds] = src[i * ss];
}
template <class R> struct FillOp {
  using Real = R;
  static constexpr int NIN = 1, UNROLL = 4;
  static constexpr bool OUT = true, ACC = false;
  const R* in[NIN];
  R fill[NIN];
  R* y;
  __device__ __forceinline__ R apply(const R (&x)[NIN], long long, Partial&) const { return x[0]; }
};

// any(l .> u)  (shiftedNormL1Box.jl:33)
template <class R> struct AnyGtOp {
  using Real = R;
  static constexpr int NIN = 2, UNROLL = 4;
  static constexpr bool OUT = false, ACC = true;
  const R* in[NIN];
  R fill[NIN];
  R* y;
  __device__ __forceinline__ R apply(const R (&x)[NIN], long long, Partial& acc) const {
    if (x[0] > x[1]) acc.bad = 1;
    return R(0);
  }
};

__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

template <class R> struct UniformOp {
  using Real = R;
  static constexpr int NIN = 1, UNROLL = 4;
  static constexpr bool OUT = true, ACC = false;
  const R* in[NIN];
  R fill[NIN];
  R* y;
  unsigned long long key;  // seed ^ (stream << 40)
  R scale, shift;
  __device__ __forceinline__ R apply(const R (&)[NIN], long long i, Partial&) const {
    unsigned long long h = splitmix64(key + (unsigned long long)i);
    R u;
    if (sizeof(R) == 8) u = (R)((double)(h >> 11) * 0x1.0p-53);
    else u = (R)((float)(h >> 40) * 0x1.0p-24f);
    return scale * u + shift;
  }
};

// Σ_i mix(word_i ^ mix(i)) mod 2^64 -- order independent, position sensitive
__global__ void __launch_bounds__(256) checksum_kernel(const unsigned long long* __restrict__ w, long long n,
                                                       unsigned long long* __restrict__ out) {
  unsigned long long acc = 0;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256)
    acc += splitmix64(w[i] ^ splitmix64((unsigned long long)i));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}

__global__ void __launch_bounds__(256) mask_kernel(const long long* __restrict__ list, long long nlist, long long n,
                                                   unsigned* __restrict__ mask) {
  for (long long j = (long long)blockIdx.x * 256 + threadIdx.x; j < nlist; j += (long long)gridDim.x * 256) {
    long long i = list[j];
    if (i >= 0 && i < n) atomicOr(mask + (i >> 5), 1u << (i & 31));
  }
}

template <class R>
static int32_t fill_impl(spx_ctx* ctx, R* p, int64_t n, R v) {
  SPX_REQUIRE(ctx != nullptr, "null context");
  SPX_REQUIRE(n >= 0 && (p != nullptr || n == 0), "bad buffer");
  DeviceGuard g(ctx->device);
  FillOp<R> op;
  op.in[0] = nullptr;
  op.fill[0] = v;
  op.y = p;
  return ew_launch(ctx, ctx->stream, op, n, 0, nullptr, nullptr);
}

template <class R>
static int32_t any_gt_impl(spx_ctx* ctx, int64_t n, const spx_bound* l, const spx_bound* u, int32_t* out) {
  SPX_REQUIRE(ctx && l && u && out, "null argument");
  SPX_REQUIRE(n >= 0, "n < 0");
  if (l->vec == nullptr && u->vec == nullptr) {
    *out = ((R)l->val > (R)u->val) ? 1 : 0;
    return SPX_OK;
  }
  DeviceGuard g(ctx->device);
  AnyGtOp<R> op;
  op.in[0] = (const R*)l->vec;
  op.in[1] = (const R*)u->vec;
  op.fill[0] = (R)l->val;
  op.fill[1] = (R)u->val;
  op.y = nullptr;
  int nb = 0;
  int32_t st = ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, &nb);
  if (st != SPX_OK) return st;
  st = finalize_partials(ctx, nb, 1, false);
  if (st != SPX_OK) return st;
  *out = ctx->h_result[0].bad > 0 ? 1 : 0;
  return SPX_OK;
}

template <class R>
static int32_t uniform_impl(spx_ctx* ctx, R* out, int64_t n, int64_t i0, uint64_t seed, uint64_t stream, R scale,
                            R shift) {
  SPX_REQUIRE(ctx != nullptr, "null context");
  SPX_REQUIRE(n >= 0 && (out != nullptr || n == 0), "bad buffer");
  DeviceGuard g(ctx->device);
  UniformOp<R> op;
  op.in[0] = nullptr;
  op.fill[0] = R(0);
  op.y = out;
  op.key = (seed ^ (stream << 40));
  op.scale = scale;
  op.shift = shift;
  return ew_launch(ctx, ctx->stream, op, n, i0, nullptr, nullptr);
}

}  // namespace spx

using namespace spx;

extern "C" {

int32_t spx_version(void) { return 100; }
const char* spx_last_error(void) { return spx::g_err; }

int32_t spx_ctx_create(spx_ctx** out, int32_t device, void* stream, int32_t own_stream) {
  SPX_REQUIRE(out != nullptr, "null out");
  *out = nullptr;
  int ndev = 0;
  SPX_CUDA(cudaGetDeviceCount(&ndev));
  SPX_REQUIRE(device >= 0 && device < ndev, "no such device");
  DeviceGuard g(device);
  cudaDeviceProp prop;
  SPX_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_error("libshiftedprox is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
    return SPX_E_UNSUPPORTED;
  }
  spx_ctx* c = new spx_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  if (own_stream == 0) {
    c->stream = (cudaStream_t)stream;  // NULL = the default stream
  } else {
    SPX_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    c->owns_stream = true;
  }
  SPX_CUDA(cudaMalloc(&c->d_partials, sizeof(Partial) * kMaxPartials * kMaxScale));
  SPX_CUDA(cudaMalloc(&c->d_result, sizeof(Partial) * kMaxScale));
  SPX_CUDA(cudaHostAlloc(&c->h_result, sizeof(Partial) * kMaxScale, cudaHostAllocDefault));
  *out = c;
  return SPX_OK;
}

int32_t spx_ctx_destroy(spx_ctx* c) {
  if (c == nullptr) return SPX_OK;
  DeviceGuard g(c->device);
  cudaStreamSynchronize(c->stream);
  for (int i = 0; i < 3; ++i)
    if (c->pipe_streams[i]) cudaStreamDestroy(c->pipe_streams[i]);
  for (cudaEvent_t ev : c->pipe_events)
    if (ev) cudaEventDestroy(ev);
  if (c->pipe_buf) cudaFree(c->pipe_buf);
  if (c->d_scratch) cudaFree(c->d_scratch);
  spx_comm_peer_detach(c);
  if (c->peer_own) cudaFree(c->peer_own);
  spx_comm_destroy(c);
  if (c->d_comm) cudaFree(c->d_comm);
  cudaFree(c->d_partials);
  cudaFree(c->d_result);
  cudaFreeHost(c->h_result);
  if (c->owns_stream) cudaStreamDestroy(c->stream);
  delete c;
  return SPX_OK;
}

int32_t spx_ctx_set_stream(spx_ctx* c, void* stream) {
  SPX_REQUIRE(c != nullptr, "null context");
  bool drained = false;
  if (c->owns_stream) {
    DeviceGuard g(c->device);
    cudaStreamSynchronize(c->stream);
    cudaStreamDestroy(c->stream);
    c->owns_stream = false;
    drained = true;  // nothing left on the old stream (which no longer exists)
  }
  // The reduction scratch (d_partials, d_result, h_result, d_scratch) is shared by every call of the context: work still
  // queued on the old stream must finish before anything enqueued on the new one touches it.
  if (!drained && (cudaStream_t)stream != c->stream) {
    DeviceGuard g(c->device);
    cudaEvent_t ev;
    SPX_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    SPX_CUDA(cudaEventRecord(ev, c->stream));
    SPX_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, ev, 0));
    SPX_CUDA(cudaEventDestroy(ev));
  }
  c->stream = (cudaStream_t)stream;
  return SPX_OK;
}

int32_t spx_ctx_synchronize(spx_ctx* c) {
  SPX_REQUIRE(c != nullptr, "null context");
  DeviceGuard g(c->device);
  SPX_CUDA(cudaStreamSynchronize(c->stream));
  return SPX_OK;
}

int32_t spx_ctx_sm_count(spx_ctx* c, int32_t* out) {
  SPX_REQUIRE(c && out, "null argument");
  *out = c->sm_count;
  return SPX_OK;
}

int32_t spx_ctx_launch_count(spx_ctx* c, int64_t* out) {
  SPX_REQUIRE(c && out, "null argument");
  *out = c->launches;
  return SPX_OK;
}

int32_t spx_malloc(spx_ctx* c, size_t bytes, void** out) {
  SPX_REQUIRE(c && out, "null argument");
  DeviceGuard g(c->device);
  *out = nullptr;
  if (bytes == 0) return SPX_OK;
  SPX_CUDA(cudaMalloc(out, bytes));
  return SPX_OK;
}
int32_t spx_free(spx_ctx* c, void* p) {
  SPX_REQUIRE(c != nullptr, "null context");
  if (p == nullptr) return SPX_OK;
  DeviceGuard g(c->device);
  SPX_CUDA(cudaStreamSynchronize(c->stream));
  SPX_CUDA(cudaFree(p));
  return SPX_OK;
}
int32_t spx_malloc_host(size_t bytes, void** out) {
  SPX_REQUIRE(out != nullptr, "null out");
  *out = nullptr;
  if (bytes == 0) return SPX_OK;
  SPX_CUDA(cudaHostAlloc(out, bytes, cudaHostAllocDefault));
  return SPX_OK;
}
int32_t spx_free_host(void* p) {
  if (p == nullptr) return SPX_OK;
  SPX_CUDA(cudaFreeHost(p));
  return SPX_OK;
}
int32_t spx_memcpy_h2d(spx_ctx* c, void* dst, const void* src, size_t bytes) {
  SPX_REQUIRE(c != nullptr, "null context");
  if (bytes == 0) return SPX_OK;
  SPX_REQUIRE(dst && src, "null buffer");
  DeviceGuard g(c->device);
  SPX_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
  // the source may be pageable and reused by the caller right away
  SPX_CUDA(cudaStreamSynchronize(c->stream));
  return SPX_OK;
}
int32_t spx_memcpy_d2h(spx_ctx* c, void* dst, const void* src, size_t bytes) {
  SPX_REQUIRE(c != nullptr, "null context");
  if (bytes == 0) return SPX_OK;
  SPX_REQUIRE(dst && src, "null buffer");
  DeviceGuard g(c->device);
  SPX_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
  SPX_CUDA(cudaStreamSynchronize(c->stream));
  return SPX_OK;
}
int32_t spx_memcpy_d2d(spx_ctx* c, void* dst, const void* src, size_t bytes) {
  SPX_REQUIRE(c != nullptr, "null context");
  if (bytes == 0 || dst == src) return SPX_OK;
  SPX_REQUIRE(dst && src, "null buffer");
  DeviceGuard g(c->device);
  SPX_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, c->stream));
  return SPX_OK;
}
int32_t spx_copy_strided(spx_ctx* c, int64_t n, int32_t elem_bytes, void* dst, int64_t dst_stride, const void* src,
                         int64_t src_stride) {
  SPX_REQUIRE(c != nullptr, "null context");
  SPX_REQUIRE(n >= 0, "n < 0");
  SPX_REQUIRE(elem_bytes == 4 || elem_bytes == 8, "element size must be 4 or 8 bytes");
  SPX_REQUIRE(dst_stride != 0 && src_stride != 0, "zero stride");
  if (n == 0) return SPX_OK;
  SPX_REQUIRE(dst && src, "null buffer");
  DeviceGuard g(c->device);
  long long want = (n + 255) / 256;
  const long long cap = (long long)c->sm_count * 8;
  const int grid = (int)(want < cap ? want : cap);
  if (elem_bytes == 8)
    spx::copy_strided_kernel<unsigned long long><<<grid, 256, 0, c->stream>>>(n, (unsigned long long*)dst, dst_stride,
                                                                         (const unsigned long long*)src, src_stride);
  else
    spx::copy_strided_kernel<unsigned><<<grid, 256, 0, c->stream>>>(n, (unsigned*)dst, dst_stride, (const unsigned*)src,
                                                               src_stride);
  c->launches++;
  SPX_CUDA(cudaGetLastError());
  return SPX_OK;
}
int32_t spx_fill_f64(spx_ctx* c, double* p, int64_t n, double v) { return fill_impl<double>(c, p, n, v); }
int32_t spx_fill_f32(spx_ctx* c, float* p, int64_t n, float v) { return fill_impl<float>(c, p, n, v); }
int32_t spx_any_gt_f64(spx_ctx* c, int64_t n, const spx_bound* l, const spx_bound* u, int32_t* out) {
  return any_gt_impl<double>(c, n, l, u, out);
}
int32_t spx_any_gt_f32(spx_ctx* c, int64_t n, const spx_bound* l, const spx_bound* u, int32_t* out) {
  return any_gt_impl<float>(c, n, l, u, out);
}

int32_t spx_build_mask(spx_ctx* c, int64_t n, const int64_t* list, int64_t nlist, uint32_t* mask) {
  SPX_REQUIRE(c && mask, "null argument");
  SPX_REQUIRE(n >= 0 && nlist >= 0 && (list != nullptr || nlist == 0), "bad list");
  DeviceGuard g(c->device);
  size_t words = (size_t)((n + 31) / 32);
  if (words) SPX_CUDA(cudaMemsetAsync(mask, 0, words * 4, c->stream));
  if (nlist > 0) {
    long long want = (nlist + 255) / 256;
    int grid = (int)(want < (long long)c->sm_count * 8 ? want : (long long)c->sm_count * 8);
    mask_kernel<<<grid, 256, 0, c->stream>>>((const long long*)list, nlist, n, mask);
    c->launches++;
    SPX_CUDA(cudaGetLastError());
  }
  return SPX_OK;
}

int32_t spx_fill_uniform_f64(spx_ctx* c, double* out, int64_t n, int64_t i0, uint64_t seed, uint64_t stream,
                             double scale, double shift) {
  return uniform_impl<double>(c, out, n, i0, seed, stream, scale, shift);
}
int32_t spx_fill_uniform_f32(spx_ctx* c, float* out, int64_t n, int64_t i0, uint64_t seed, uint64_t stream,
                             float scale, float shift) {
  return uniform_impl<float>(c, out, n, i0, seed, stream, scale, shift);
}

int32_t spx_checksum(spx_ctx* c, const void* p, int64_t nwords, uint64_t* out) {
  SPX_REQUIRE(c && out, "null argument");
  SPX_REQUIRE(nwords >= 0 && (p != nullptr || nwords == 0), "bad buffer");
  DeviceGuard g(c->device);
  int32_t st = ensure_scratch(c, 4096);
  if (st != SPX_OK) return st;
  SPX_CUDA(cudaMemsetAsync(c->d_scratch, 0, 8, c->stream));
  if (nwords > 0) {
    long long want = (nwords + 255) / 256;
    int grid = (int)(want < (long long)c->sm_count * 8 ? want : (long long)c->sm_count * 8);
    checksum_kernel<<<grid, 256, 0, c->stream>>>((const unsigned long long*)p, nwords,
                                                 (unsigned long long*)c->d_scratch);
    c->launches++;
    SPX_CUDA(cudaGetLastError());
  }
  SPX_CUDA(cudaMemcpyAsync(out, c->d_scratch, 8, cudaMemcpyDeviceToHost, c->stream));
  SPX_CUDA(cudaStreamSynchronize(c->stream));
  return SPX_OK;
}

double spx_prox_zero_f64(double q, double l, double u) { return prox_zero<double>(q, l, u); }
double spx_iprox_zero_f64(double d, double g, double l, double u) { return iprox_zero<double>(d, g, l, u); }
float spx_prox_zero_f32(float q, float l, float u) { return prox_zero<float>(q, l, u); }
float spx_iprox_zero_f32(float d, float g, float l, float u) { return iprox_zero<float>(d, g, l, u); }

}  // extern "C"
