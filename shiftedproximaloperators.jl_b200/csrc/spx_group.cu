// spx_group.cu -- group-norm operators: segmented sub-warp reductions.
//
// A warp walks over tasks of 32 consecutive groups.  Inside a task it packs as many groups as fit
// into one ROUND: 2^j groups of L = 32 / 2^j lanes each, L the smallest power of two such that every
// group of the round holds at most 8 L elements (8 elements per lane stay in registers for the whole
// prox: one HBM read per operand, one write).  Groups of 64 run four to a warp, groups of <= 8
// thirty-two to a warp, so the per-group scalar work -- the norm, and for the Binf form the whole root
// search -- is shared by the groups of a round instead of being repeated on 32 idle lanes.  Groups of
// more than 256 elements take the whole warp, stash `sol` in the output vector and re-read it through
// L1/L2; they run in a second launch of the same kernel (PART = 1) so that the register-resident rounds
// and the deeply batched loads a lone warp needs to hide latency do not share one register budget.  Sums of squares are accumulated in Float64 whatever R is; the butterfly order is fixed, so
// results are deterministic.
#include <algorithm>
#include <cstddef>

#include "spx_elementwise.cuh"
#include "spx_ops.cuh"

namespace spx {

constexpr int kGroupThreads = 256;
constexpr int kEPL = 8;    // elements per lane kept in registers
constexpr int kTask = 32;  // consecutive groups per warp task
// groups of kBigMin < m <= kBigMax elements take a whole CTA: 16 elements per thread in registers, one HBM
// read per operand like the short groups (the warp path would stash and re-read them)
constexpr long long kBigMin = 1024, kBigMax = 4096;
constexpr int kBigE = (int)(kBigMax / kGroupThreads);
// CTA-per-group classes of ShiftedGroupNormL2: (kMidMin, kBigMin] with 128 threads, (kBigMin, kBigMax] with 256
constexpr long long kMidMin = 256;
// `classes`: which of them have their kernel launched in this call (bit 0: the 128-thread class, bit 1: the 256-thread
// one); the warp kernels take every long group that is in none of the launched classes
__device__ __forceinline__ bool in_launched_class(long long m, unsigned classes) {
  return ((classes & 1u) != 0u && m > kMidMin && m <= kBigMin) || ((classes & 2u) != 0u && m > kBigMin && m <= kBigMax);
}

#ifdef SPX_GROUP_STATS
__device__ unsigned long long g_stat_evals = 0, g_stat_groups = 0, g_stat_big[3] = {0, 0, 0};  // big: evals, groups, rejected
#endif

template <class R> __device__ __forceinline__ R ldv(const R* p) {
  Pack<R, 1> t;
  ld_stream(p, t);
  return t.v[0];
}
template <class R> __device__ __forceinline__ void stv(R* p, R v) {
  Pack<R, 1> t;
  t.v[0] = v;
  st_stream(p, t);
}

// reference form (shiftedGroupNormL2Binf.jl:83): sign(x) max(0, |x| - a)
template <class R> __device__ __forceinline__ R softthres(R x, R a) {
  return jl_sign(x) * jl_max(R(0), jl_abs(x) - a);
}
// bit-identical to the reference form, NaNs included (`!(a <= 0)` keeps a NaN threshold excess):
// sign(±0) max(0, -a) = ±0 = copysign(0, ±0), sign(NaN) = NaN = copysign(NaN, NaN)
__device__ __forceinline__ double softthres_sel(double x, double a) {
  const double ex = fabs(x) - a;
  return copysign(!(ex <= 0.0) ? ex : 0.0, x);
}
__device__ __forceinline__ float softthres_sel(float x, float a) {
  const float ex = fabsf(x) - a;
  return copysignf(!(ex <= 0.0f) ? ex : 0.0f, x);
}
// same value for non-NaN operands, three instructions (used inside the root search only)
__device__ __forceinline__ double softthres_fast(double x, double a) { return copysign(fmax(fabs(x) - a, 0.0), x); }
__device__ __forceinline__ float softthres_fast(float x, float a) { return copysignf(fmaxf(fabsf(x) - a, 0.0f), x); }

// a / b to ~1 ulp for normal operands (reciprocal seed + two Newton steps + one residual correction);
// anything else yields Inf/NaN, which every caller treats as "no usable candidate"
__device__ __forceinline__ double div_fast(double a, double b) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(b));
  double e = __fma_rn(-b, y, 1.0);
  y = __fma_rn(y, e, y);
  e = __fma_rn(-b, y, 1.0);
  y = __fma_rn(y, e, y);
  const double q = a * y;
  const double r = __fma_rn(-b, q, a);
  return __fma_rn(r, y, q);
}
__device__ __forceinline__ float div_fast(float a, float b) { return a / b; }

// sum over the L lanes of a group (L a power of two, lanes aligned); every lane gets the total.
// L is uniform over the warp: the switch is a uniform branch into a fully unrolled butterfly.
template <int L> __device__ __forceinline__ void sub_sum_t(double& v, double& w) {
#pragma unroll
  for (int o = L >> 1; o > 0; o >>= 1) {
    v += __shfl_xor_sync(0xffffffffu, v, o);
    w += __shfl_xor_sync(0xffffffffu, w, o);
  }
}
__device__ __forceinline__ void sub_sum2(double& v, double& w, int L) {
  switch (L) {
    case 32: sub_sum_t<32>(v, w); break;
    case 16: sub_sum_t<16>(v, w); break;
    case 8: sub_sum_t<8>(v, w); break;
    case 4: sub_sum_t<4>(v, w); break;
    case 2: sub_sum_t<2>(v, w); break;
    default: break;
  }
}
__device__ __forceinline__ double sub_sum(double v, int L) {
  for (int o = L >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Next task of a warp: round-robin (deterministic: required when ψ(y) partial sums ride along), or, when the
// tasks are very unequal and heavy (the Binf root search on long groups) and nothing order-dependent is
// accumulated, one task at a time from a global counter.
__device__ __forceinline__ long long next_task(long long cur, long long nwarps, unsigned long long* counter,
                                               int lane) {
  if (counter == nullptr) return cur + nwarps;
  unsigned long long t = 0;
  if (lane == 0) t = atomicAdd(counter, 1ull);
  return (long long)__shfl_sync(0xffffffffu, t, 0);
}

// ---- round planning ----------------------------------------------------------------------------
// le[k] bit j: group j of the task has at most 8 << k elements (k = 0..5).  Returns k such that the
// round holds 32 >> k groups of 1 << k lanes, or -1 when the group at `pos` is a long one.
__device__ __forceinline__ int plan_round(const unsigned (&le)[6], int pos) {
#pragma unroll
  for (int k = 0; k <= 5; ++k) {
    const int c = 32 >> k;
    const unsigned need = (c >= 32 ? 0xffffffffu : ((1u << c) - 1u)) << pos;
    if ((le[k] & need) == need) return k;
  }
  return -1;
}

struct TaskHead {
  long long lo, hi;  // lane j: offsets of group g0 + j (0, 0 beyond the task)
  unsigned le[6];
  int cnt;
};
__device__ __forceinline__ TaskHead load_task(const long long* __restrict__ offs, long long g0, long long ngroups,
                                              int lane) {
  TaskHead t;
  const long long left = ngroups - g0;
  t.cnt = left < kTask ? (int)left : kTask;
  t.lo = 0;
  t.hi = 0;
  if (lane < t.cnt) {
    t.lo = offs[g0 + lane];
    t.hi = offs[g0 + lane + 1];
  }
  const long long m = t.hi - t.lo;
#pragma unroll
  for (int k = 0; k <= 5; ++k) t.le[k] = __ballot_sync(0xffffffffu, m <= ((long long)kEPL << k));
  return t;
}

// the part of a group a lane holds during a round
// KEEP_XS: xk + sj stays in registers (the one-pass GroupNormL2); the Binf form, which holds the tile
// through a root search, drops it and re-reads sj (an L2 hit) when it writes the result
template <class R, bool KEEP_XS> struct Tile {
  R sol[kEPL], xkr[kEPL], xs[KEEP_XS ? kEPL : 1];
  long long b, e;  // the lane's group (b == e: none)
  int L, sub;
  bool valid;
  // SHIFTED = false: xk == sj == NULL, the shifts read as zeros (unshifted GroupNormL2 prox!, groupNormL2.jl:41-58)
  template <bool SHIFTED = true>
  __device__ __forceinline__ void load(const TaskHead& t, int k, int pos, int lane, const R* xk, const R* sj,
                                       const R* q) {
    L = 1 << k;
    sub = lane & (L - 1);
    const int gi = pos + (lane >> k);
    const long long lo = __shfl_sync(0xffffffffu, t.lo, gi & 31);
    const long long hi = __shfl_sync(0xffffffffu, t.hi, gi & 31);
    valid = gi < t.cnt;
    b = valid ? lo : 0;
    e = valid ? hi : 0;
#pragma unroll
    for (int j = 0; j < kEPL; ++j) {
      const long long i = b + (long long)j * L + sub;
      sol[j] = R(0);
      xkr[j] = R(0);
      if (KEEP_XS) xs[j] = R(0);
      if (i < e) {
        const R xi = SHIFTED ? ldv(xk + i) : R(0), si = SHIFTED ? ldv(sj + i) : R(0), qi = ldv(q + i);
        sol[j] = (qi + xi) + si;  // shiftedGroupNormL2.jl:65, shiftedGroupNormL2Binf.jl:80
        xkr[j] = xi;
        if (KEEP_XS) xs[j] = xi + si;
      }
    }
  }
  __device__ __forceinline__ int group_in_task(int pos, int k, int lane) const { return pos + (lane >> k); }
};

// ------------------------------------------------------- ShiftedGroupNormL2 --
// shiftedGroupNormL2.jl:52-79
// Loads are batched four iterations deep before anything is stored: y may alias q, so the compiler
// cannot hoist them itself, and a warp that owns a long group is alone in hiding its latency.
// STEP (the solver step, spx_step_groupl2): y = s, q = ∇f read as q = (-ν)∇f rounded to R (mnu = -ν); the second loop
// re-reads ∇f beside the stash, also writes xsy = (xk + sj) + s (when given) and adds Σ s² and Σ ∇f·s of the lane's
// elements to ss2 and dot.  s overlaps none of xk, sj, ∇f (the alias rule of the group steps), so stashing sol in s is
// safe; xsy may be xk or sj: every element is read before the same lane writes it.
template <class R, bool PSI, bool SHIFTED, bool STEP = false>
__device__ __forceinline__ double l2_long_group(R* y, const R* xk, const R* sj, const R* q, long long b, long long e,
                                                R lam, R sigma, int lane, R* xsy = nullptr, R mnu = R(0),
                                                double* ss2 = nullptr, double* dot = nullptr) {
  double ss = 0.0;
  for (long long i0 = b + lane; i0 < e; i0 += 128) {
    R xv[4], sv[4], qv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long i = i0 + 32 * u;
      if (i < e) {
        xv[u] = SHIFTED ? ldv(xk + i) : R(0);
        sv[u] = SHIFTED ? ldv(sj + i) : R(0);
        qv[u] = ldv(q + i);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long i = i0 + 32 * u;
      if (i < e) {
        if constexpr (STEP) qv[u] = mnu * qv[u];  // q = -ν ∇f
        const R s = (qv[u] + xv[u]) + sv[u];
        y[i] = s;  // stash sol (each lane re-reads only what it wrote)
        ss += (double)s * (double)s;
      }
    }
  }
  ss = warp_sum(ss);
  const R snorm = (R)sqrt(ss);
  const R alpha = jl_max(R(1) - sigma * lam / snorm, R(0));
  double vv = 0.0;
  for (long long i0 = b + lane; i0 < e; i0 += 128) {
    R xv[4], sv[4], yv[4], gv[STEP ? 4 : 1];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long i = i0 + 32 * u;
      if (i < e) {
        xv[u] = SHIFTED ? xk[i] : R(0);
        sv[u] = SHIFTED ? sj[i] : R(0);
        yv[u] = y[i];
        if constexpr (STEP) gv[u] = q[i];
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long i = i0 + 32 * u;
      if (i < e) {
        const R xsi = xv[u] + sv[u];
        const R o = (snorm == R(0) ? R(0) : alpha * yv[u]) - xsi;
        stv(y + i, o);
        if constexpr (STEP) {
          const R v = xsi + o;  // ψ's own argument (ShiftedProximalOperators.jl:52)
          if (xsy != nullptr) stv(xsy + i, v);
          vv += (double)v * (double)v;
          *ss2 = __fma_rn((double)o, (double)o, *ss2);
          *dot = __fma_rn((double)gv[u], (double)o, *dot);
        } else if (PSI) {
          const double v = (double)(xsi + o);
          vv += v * v;
        }
      }
    }
  }
  if (PSI) vv = warp_sum(vv);
  // unshifted GroupNormL2.prox! returns Σ λ_g ‖x_g‖ -- the norms of its INPUT (groupNormL2.jl:49-54)
  return (PSI && !SHIFTED) ? ss : vv;
}

// PART 0: groups of <= 256 elements, 1: the longer ones; SHIFTED = false: xk == sj == NULL
// STEP (PART 1 only, PSI and SHIFTED): the long groups of the solver step (l2_long_group), q = ∇f; slot 0 is
// partials[blockIdx.x] = {ψ, Σ s², -1}, slot 1 part1[blockIdx.x] = {Σ ∇f·s, 0, -1}
template <class R, bool PSI, int PART, bool SHIFTED, bool STEP = false>
__global__ void __launch_bounds__(kGroupThreads)
    group_l2_kernel(R* y, const R* xk, const R* sj, const R* q, long long ngroups,
                    const long long* __restrict__ offs, const R* __restrict__ lambda_g, R sigma, unsigned classes,
                    Partial* __restrict__ partials, R* xsy, R mnu, Partial* __restrict__ part1) {
  static_assert(!STEP || (PSI && PART == 1 && SHIFTED), "the step form takes the shifted long groups");
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * kGroupThreads + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * kGroupThreads) >> 5;
  const long long ntasks = (ngroups + kTask - 1) / kTask;
  double psi = 0.0, ss2 = 0.0, dot = 0.0;
  for (long long task = warp; task < ntasks; task += nwarps) {
    const long long g0 = task * kTask;
    const TaskHead th = load_task(offs, g0, ngroups, lane);
    // le[5]: groups of <= 256 elements (lanes beyond the task count as such)
    if (PART == 1 ? (th.le[5] == 0xffffffffu) : (th.le[5] == 0u)) continue;
    const R lam_lane = lane < th.cnt ? lambda_g[g0 + lane] : R(0);
    int pos = 0;
    while (pos < th.cnt) {
      const int k = plan_round(th.le, pos);
      if (k < 0) {  // long group: the whole warp (a whole CTA of group_l2_big_kernel for 1024 < m <= 4096)
        if (PART == 1) {
          const long long b = __shfl_sync(0xffffffffu, th.lo, pos), e = __shfl_sync(0xffffffffu, th.hi, pos);
          if (!in_launched_class(e - b, classes)) {
            const R lam = __shfl_sync(0xffffffffu, lam_lane, pos);
            const double vv =
                l2_long_group<R, PSI, SHIFTED, STEP>(y, xk, sj, q, b, e, lam, sigma, lane, xsy, mnu, &ss2, &dot);
            if (PSI && lane == 0) psi += (double)(lam * (R)sqrt(vv));  // λ_g ‖v_g‖  groupNormL2.jl:36
          }
        }
        pos += 1;
        continue;
      }
      if (PART == 1) {
        pos += 32 >> k;
        continue;
      }
      Tile<R, true> t;
      t.template load<SHIFTED>(th, k, pos, lane, xk, sj, q);
      const R lam = __shfl_sync(0xffffffffu, lam_lane, t.group_in_task(pos, k, lane) & 31);
      double ss = 0.0;
#pragma unroll
      for (int j = 0; j < kEPL; ++j) ss += (double)t.sol[j] * (double)t.sol[j];
      ss = sub_sum(ss, t.L);
      const R snorm = (R)sqrt_fast(ss);
      const R alpha = jl_max(R(1) - sigma * lam / snorm, R(0));
      double vv = 0.0;
#pragma unroll
      for (int j = 0; j < kEPL; ++j) {
        const long long i = t.b + (long long)j * t.L + t.sub;
        if (i < t.e) {
          const R o = (snorm == R(0) ? R(0) : alpha * t.sol[j]) - t.xs[j];  // :70-77
          stv(y + i, o);
          if (PSI) {
            const double v = (double)(t.xs[j] + o);
            vv += v * v;
          }
        }
      }
      if (PSI) {
        vv = sub_sum(vv, t.L);
        // shifted: λ_g ‖(xk + sj + y)_g‖; unshifted (xk == NULL): λ_g ‖x_g‖ of the input, as groupNormL2.jl:49-54
        if (t.valid && t.sub == 0) psi += (double)(lam * (SHIFTED ? (R)sqrt_fast(vv) : snorm));
      }
      pos += 32 >> k;
    }
  }
  if constexpr (STEP) {
    Partial p{psi, ss2, -1}, p2{dot, 0.0, -1};
    p = block_fold<kGroupThreads>(p);
    p2 = block_fold<kGroupThreads>(p2);
    if (threadIdx.x == 0) {
      partials[blockIdx.x] = p;
      part1[blockIdx.x] = p2;
    }
  } else if (PSI) {
    Partial p;
    p.s = psi;
    p.s2 = 0.0;
    p.bad = -1;
    p = block_fold<kGroupThreads>(p);
    if (threadIdx.x == 0) partials[blockIdx.x] = p;
  }
}

// ---- one CTA per group of 1025..4096 elements ------------------------------------------------------
// Every CTA scans chunks of 256 groups (grid-stride), lists the big ones in index order and takes them one
// after the other: 16 elements per thread in registers (all 48 loads of a thread in flight at once), one block
// reduction for the norm, y written once.
template <int T = kGroupThreads> __device__ __forceinline__ double block_sum(double v, double* red) {
  v = warp_sum(v);
  __syncthreads();  // red reuse
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
#pragma unroll
  for (int w = 0; w < T / 32; ++w) t += red[w];
  return t;
}
// L2 prefetch of elements [b, e) of up to three operand vectors by the whole CTA (T threads): a CTA-per-group kernel
// issues this for its NEXT group right after the loads of the current one, so the next load phase finds its lines in L2
// instead of paying HBM latency with nothing else in flight.
template <class R, int T>
__device__ __forceinline__ void prefetch_group_l2(const R* p0, const R* p1, const R* p2, long long b, long long e) {
  const R* ps[3] = {p0, p1, p2};
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    if (ps[a] == nullptr) continue;
    const uintptr_t lo = (uintptr_t)(ps[a] + b) & ~(uintptr_t)127, hi = (uintptr_t)(ps[a] + e);
    for (uintptr_t l = lo + (uintptr_t)threadIdx.x * 128u; l < hi; l += (uintptr_t)T * 128u)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(l));
  }
}

// ---- TMA bulk copies (cp.async.bulk, one elected thread) for the CTA-per-group classes -------------------------------
// A group is a contiguous run of each operand vector, so one thread moves it with three bulk copies that complete on an
// mbarrier: no LSU instructions, no registers, any thread may read any element afterwards.  Bulk copies want 16-byte
// aligned addresses and sizes while a group starts on an element boundary: the copy starts at the 16-byte granule that
// holds the first element and ends with the granule that holds the last one (the few neighbouring bytes of the same
// granules are read and ignored -- a granule that holds a valid byte lies in the same page); `skip` elements of
// padding result at the front of each plane, per operand.  The copy primitives (bulk_g2s, mbar_*) are in spx_common.cuh.
template <class R> __device__ __forceinline__ int bulk_skip(const R* p) {  // elements of front padding in the plane
  return (int)(((uintptr_t)p & 15u) / sizeof(R));
}
// elements per staging plane of a class of groups of up to `maxm` elements (the padding of both ends included)
template <class R> __host__ __device__ constexpr int bulk_plane(int maxm) { return maxm + 2 * (int)(16 / sizeof(R)); }
// called by ONE thread: group [b, e) of NP operands into planes of PLS elements, completion on `bar`
template <class R, int NP, int PLS>
__device__ __forceinline__ void stage_group_bulk(R* stage, uint64_t* bar, const R* q, const R* xk, const R* sj, long long b,
                                                 long long e) {
  const R* ps[3] = {q, xk, sj};
  uintptr_t lo[NP];
  uint32_t bytes[NP], total = 0;
#pragma unroll
  for (int a = 0; a < NP; ++a) {
    lo[a] = (uintptr_t)(ps[a] + b) & ~(uintptr_t)15;
    bytes[a] = (uint32_t)((((uintptr_t)(ps[a] + e) + 15u) & ~(uintptr_t)15) - lo[a]);
    total += bytes[a];
  }
  mbar_expect_tx(bar, total);
#pragma unroll
  for (int a = 0; a < NP; ++a) bulk_g2s(stage + a * PLS, (const void*)lo[a], bytes[a], bar);
}

// index-ordered list of one chunk's (T groups) members of the class LO < m <= HI; returns how many
template <int T, int LO, int HI>
__device__ __forceinline__ int list_class_groups(const long long* __restrict__ offs, long long g0, long long ngroups,
                                                 int* list, int* wcount) {
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const long long g = g0 + t;
  const long long m = g < ngroups ? offs[g + 1] - offs[g] : 0;
  const bool big = m > LO && m <= HI;
  const unsigned bal = __ballot_sync(0xffffffffu, big);
  __syncthreads();  // list / wcount reuse
  if (lane == 0) wcount[w] = __popc(bal);
  __syncthreads();
  int base = 0, total = 0;
#pragma unroll
  for (int ww = 0; ww < T / 32; ++ww) {
    if (ww < w) base += wcount[ww];
    total += wcount[ww];
  }
  if (big) list[base + __popc(bal & ((1u << lane) - 1u))] = t;
  __syncthreads();
  return total;
}

// ST staging buffers of NP planes (PLS elements each) that take a chunk's listed groups in list order: listed group j
// lands in buffer j % ST, and thread 0 refills that buffer with group j + ST once every thread holds group j.  `bar`
// (ST mbarriers) and `buf` are the kernel's shared memory; the constructor initialises the mbarriers.
template <class R, int NP, int PLS, int ST> struct StageRing {
  uint64_t* bar;
  R* buf;
  uint32_t phases;  // bit s: the parity buffer s completes next
  int cur;          // the buffer `wait` returned last
  __device__ __forceinline__ StageRing(uint64_t* bar_, R* buf_) : bar(bar_), buf(buf_) {
    if (threadIdx.x == 0)
      for (int s = 0; s < ST; ++s) mbar_init(&bar[s], 1);
    __syncthreads();
    phases = 0;
  }
  // thread 0: the copies of the first ST listed groups
  __device__ __forceinline__ void prime(const int* list, int nlisted, long long g0, const long long* __restrict__ offs,
                                        const R* p0, const R* p1, const R* p2) {
    if (threadIdx.x != 0) return;
    fence_proxy_async();
    for (int s = 0; s < ST && s < nlisted; ++s) {
      const long long g = g0 + list[s];
      stage_group_bulk<R, NP, PLS>(buf + s * NP * PLS, &bar[s], p0, p1, p2, offs[g], offs[g + 1]);
    }
  }
  // the planes of listed group j, once its copies have landed
  __device__ __forceinline__ R* wait(int j) {
    cur = j % ST;
    mbar_wait(&bar[cur], (phases >> cur) & 1u);
    phases ^= 1u << cur;
    return buf + cur * NP * PLS;
  }
  // [b, e) of listed group j + ST; false when the list ends before it
  __device__ __forceinline__ bool ahead(const int* list, int nlisted, int j, long long g0,
                                        const long long* __restrict__ offs, long long& b, long long& e) const {
    if (j + ST >= nlisted) return false;
    const long long g = g0 + list[j + ST];
    b = offs[g];
    e = offs[g + 1];
    return true;
  }
  // thread 0, once every thread holds the group `wait` returned: its buffer takes group [b, e) (the one `ahead` gave)
  __device__ __forceinline__ void refill(const R* p0, const R* p1, const R* p2, long long b, long long e) {
    fence_proxy_async();
    stage_group_bulk<R, NP, PLS>(buf + cur * NP * PLS, &bar[cur], p0, p1, p2, b, e);
  }
};

// one group of a CTA-per-group class, E elements per thread (E T >= m); returns the group's ψ term.  The group has
// been bulk-copied into `stage`, the buffer of `ring` waited on last; once every thread holds its elements in registers (the
// barrier of the first block sum) thread 0 refills the buffer with [nb, ne), the group ST places further down the list,
// so that group's HBM latency is spent under the work on the ST - 1 groups in between (ST = 1: under this group's
// scaling and stores).
// STEP (the solver step): the q plane holds ∇f and q = (-ν)∇f is rounded to R as it is read (mnu = -ν); the store loop
// also writes xsy = (xk + sj) + s (when given) and adds Σ s² and Σ ∇f·s of the thread's elements to ss2 and dot.  The
// store loop reads ∇f from the stage again, so the buffer is refilled only after the block sum of ψ (∇f held in
// registers, or re-read from global memory, needs more registers still).
template <class R, bool PSI, bool SHIFTED, int E, int T, int PLS, bool STEP = false, class Ring>
__device__ __forceinline__ double l2_big_group(R* y, const R* xk, const R* sj, const R* q, long long b, long long e, R lam,
                                               R sigma, double* red, const R* stage, Ring& ring, long long nb,
                                               long long ne, R* xsy = nullptr, R mnu = R(0), double* ss2 = nullptr,
                                               double* dot = nullptr) {
  const int t = threadIdx.x;
  R sol[E], xs[E];
  double ss = 0.0;
  const R* pq = stage + bulk_skip(q + b) + t;
  const R* px = stage + PLS + bulk_skip(xk + b) + t;
  const R* pj = stage + 2 * PLS + bulk_skip(sj + b) + t;
#pragma unroll
  for (int k = 0; k < E; ++k) {
    const long long i = b + (long long)k * T + t;
    sol[k] = R(0);
    xs[k] = R(0);
    if (i < e) {
      const R xi = SHIFTED ? px[k * T] : R(0), si = SHIFTED ? pj[k * T] : R(0);
      const R qi = STEP ? mnu * pq[k * T] : pq[k * T];  // STEP: q = -ν ∇f
      sol[k] = (qi + xi) + si;  // shiftedGroupNormL2.jl:65
      xs[k] = xi + si;
      ss += (double)sol[k] * (double)sol[k];
    }
  }
  ss = block_sum<T>(ss, red);
  if (!STEP && t == 0 && ne > nb) ring.refill(q, xk, sj, nb, ne);
  const R snorm = (R)sqrt(ss);
  const R alpha = jl_max(R(1) - sigma * lam / snorm, R(0));
  double vv = 0.0;
  if constexpr (STEP) {
#pragma unroll
    for (int k = 0; k < E; ++k) {
      const long long i = b + (long long)k * T + t;
      if (i < e) {
        const R gk = pq[k * T];
        const R o = (snorm == R(0) ? R(0) : alpha * sol[k]) - xs[k];  // :70-77
        stv(y + i, o);
        const R v = xs[k] + o;  // ψ's own argument (ShiftedProximalOperators.jl:52)
        if (xsy != nullptr) stv(xsy + i, v);
        vv += (double)v * (double)v;
        *ss2 = __fma_rn((double)o, (double)o, *ss2);
        *dot = __fma_rn((double)gk, (double)o, *dot);
      }
    }
  } else {
#pragma unroll
    for (int k = 0; k < E; ++k) {
      const long long i = b + (long long)k * T + t;
      if (i < e) {
        const R o = (snorm == R(0) ? R(0) : alpha * sol[k]) - xs[k];  // :70-77
        stv(y + i, o);
        if (PSI) {
          const double v = (double)(xs[k] + o);
          vv += v * v;
        }
      }
    }
  }
  if (!PSI) return 0.0;
  vv = block_sum<T>(vv, red);
  if (STEP && t == 0 && ne > nb) ring.refill(q, xk, sj, nb, ne);  // every thread has read its ∇f from the stage
  // shifted: λ_g ‖(xk + sj + y)_g‖; unshifted: λ_g ‖x_g‖ of the input (groupNormL2.jl:49-54)
  return (double)(lam * (SHIFTED ? (R)sqrt(vv) : snorm));
}

// T threads per group of LO < m <= EB T elements (EA per thread up to EA T elements, EB above); ST staging buffers
// STEP (PSI and SHIFTED): the solver step, q = ∇f (see l2_big_group); slot 0 is partials[blockIdx.x] = {ψ, Σ s², -1},
// slot 1 part1[blockIdx.x] = {Σ ∇f·s, 0, -1}.  With 256 threads the STEP form runs one CTA per SM fewer than the prox!
// form (Float32 3 -> 2, Float64 2 -> 1), the occupancy at which it does not spill.
template <class R, bool PSI, bool SHIFTED, int T, int LO, int EA, int EB, int ST, bool STEP = false>
__global__ void __launch_bounds__(T, (sizeof(R) == 4 ? 3 : 2) * 256 / T - (STEP && T == 256 ? 1 : 0))
    group_l2_big_kernel(R* y, const R* xk, const R* sj, const R* q, long long ngroups,
                        const long long* __restrict__ offs, const R* __restrict__ lambda_g, R sigma,
                        Partial* __restrict__ partials, R* xsy, R mnu, Partial* __restrict__ part1) {
  static_assert(!STEP || (PSI && SHIFTED), "the step form is the shifted one with ψ");
  constexpr int PLS = bulk_plane<R>(EB * T), NP = SHIFTED ? 3 : 1;
  __shared__ int list[T];
  __shared__ int wcount[T / 32];
  __shared__ double red[T / 32];
  __shared__ __align__(8) uint64_t bar[ST];
  extern __shared__ __align__(128) unsigned char l2_stage_raw[];
  const int t = threadIdx.x;
  StageRing<R, NP, PLS, ST> ring(bar, reinterpret_cast<R*>(l2_stage_raw));  // q | xk | sj
  double psi = 0.0, ss2 = 0.0, dot = 0.0;
  for (long long g0 = (long long)blockIdx.x * T; g0 < ngroups; g0 += (long long)gridDim.x * T) {
    const int nbig = list_class_groups<T, LO, EB * T>(offs, g0, ngroups, list, wcount);
    ring.prime(list, nbig, g0, offs, q, xk, sj);
    for (int j = 0; j < nbig; ++j) {
      const long long g = g0 + list[j];
      const long long b = offs[g], e = offs[g + 1];
      const R lam = lambda_g[g];
      long long nb = 0, ne = 0;
      ring.ahead(list, nbig, j, g0, offs, nb, ne);
      const R* const stage = ring.wait(j);
      double term;
      if (e - b <= EA * T)
        term = l2_big_group<R, PSI, SHIFTED, EA, T, PLS, STEP>(y, xk, sj, q, b, e, lam, sigma, red, stage, ring, nb, ne,
                                                               xsy, mnu, &ss2, &dot);
      else
        term = l2_big_group<R, PSI, SHIFTED, EB, T, PLS, STEP>(y, xk, sj, q, b, e, lam, sigma, red, stage, ring, nb, ne,
                                                               xsy, mnu, &ss2, &dot);
      if (PSI && t == 0) psi += term;
    }
  }
  if constexpr (STEP) {
    Partial p{t == 0 ? psi : 0.0, ss2, -1}, p2{dot, 0.0, -1};
    p = block_fold<T>(p);
    p2 = block_fold<T>(p2);
    if (t == 0) {
      partials[blockIdx.x] = p;
      part1[blockIdx.x] = p2;
    }
  } else if (PSI && t == 0) {
    Partial p;
    p.s = psi;
    p.s2 = 0.0;
    p.bad = -1;
    partials[blockIdx.x] = p;
  }
}

// --------------------------------------------------- ShiftedGroupNormL2Binf --
// shiftedGroupNormL2Binf.jl:67-119.  The views give the root search Σ f(sol_i, sol_i/σ, xk_i)² over
// the lane's group: from registers (a round of short groups) or from the stash (a long group).
// One element of froot's sum, (σ softthres(sol/σ - c xk, Δc) - sol)², in the equivalent form
// (S(sol - σc xk, σΔc) - sol)², S the soft threshold: no division, and the thresholded case is a
// select.  Fused multiply-adds are fine here: the search only needs the sign change of froot, whose
// rounding noise differs between any two summation orders anyway.
// Also accumulates Σ w_i dw_i/d(σc) (dw/d(σc) = -xk - Δ sign(t) on the entries the threshold keeps, 0 on the
// others), which gives froot'(n) for the Newton steps of the search.
__device__ __forceinline__ void froot_term(double so, double xg, double sc, double sdc, double delta, double& ss,
                                           double& dot) {
  const double t = __fma_rn(-sc, xg, so);
  const double a = fabs(t) - sdc;
  const double z = copysign(a, t) - so;
  const bool act = a > 0.0;
  const double w = act ? z : so;
  const double dw = act ? (-xg - copysign(delta, t)) : 0.0;
  ss = __fma_rn(w, w, ss);
  dot = __fma_rn(w, dw, dot);
}
__device__ __forceinline__ void froot_term(float so, float xg, float sc, float sdc, float delta, double& ss,
                                           double& dot) {
  const float t = fmaf(-sc, xg, so);
  const float a = fabsf(t) - sdc;
  const float z = copysignf(a, t) - so;
  const bool act = a > 0.0f;
  const double w = (double)(act ? z : so);
  const double dw = (double)(act ? (-xg - copysignf(delta, t)) : 0.0f);
  ss = __fma_rn(w, w, ss);
  dot = __fma_rn(w, dw, dot);
}

template <class R, class TileT = Tile<R, false>> struct TileView {
  const TileT& t;
  UDiv<R> by_sigma;
  // Σ f(sol_i, sol_i/σ, xk_i)² over the lane's group
  template <class F> __device__ __forceinline__ double sumsq(F f) const {
    double ss = 0.0;
#pragma unroll
    for (int j = 0; j < kEPL; ++j) {
      const double w = (double)f(t.sol[j], by_sigma(t.sol[j]), t.xkr[j]);
      ss = __fma_rn(w, w, ss);
    }
    return sub_sum(ss, t.L);
  }
  // Σ (σ softthres(sol/σ - step xk, Δ step))² = Σ S(sol - σ step xk, σ Δ step)² (division-free: lmax is only a
  // bracket end), Σ sol², Σ xk²; sstep = σ step, sdstep = σ Δ step
  __device__ __forceinline__ void norms(R sstep, R sdstep, double& z2, double& s2, double& x2) const {
#pragma unroll
    for (int j = 0; j < kEPL; ++j) {
      const double z = (double)softthres_fast(t.sol[j] - sstep * t.xkr[j], sdstep);
      z2 = __fma_rn(z, z, z2);
      s2 = __fma_rn((double)t.sol[j], (double)t.sol[j], s2);
      x2 = __fma_rn((double)t.xkr[j], (double)t.xkr[j], x2);
    }
    sub_sum2(z2, s2, t.L);
    x2 = sub_sum(x2, t.L);
  }
  __device__ __forceinline__ double froot_sum(R sc, R sdc, R delta, double& dot) const {
    double s0 = 0.0, s1 = 0.0, d0 = 0.0, d1 = 0.0;
#pragma unroll
    for (int j = 0; j < kEPL; j += 2) {
      froot_term(t.sol[j], t.xkr[j], sc, sdc, delta, s0, d0);
      froot_term(t.sol[j + 1], t.xkr[j + 1], sc, sdc, delta, s1, d1);
    }
    double ss = s0 + s1;
    dot = d0 + d1;
    sub_sum2(ss, dot, t.L);
    return ss;
  }
};
template <class R> struct LongView {
  const R* ysol;  // stashed sol (y)
  const R* xk;
  long long b, e;
  int lane;
  UDiv<R> by_sigma;
  template <class F> __device__ __forceinline__ double sumsq(F f) const {
    double ss = 0.0;
    for (long long i0 = b + lane; i0 < e; i0 += 128) {
      R so[4], xg[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const long long i = i0 + 32 * u;
        so[u] = i < e ? ysol[i] : R(0);
        xg[u] = i < e ? xk[i] : R(0);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const double w = (i0 + 32 * u < e) ? (double)f(so[u], by_sigma(so[u]), xg[u]) : 0.0;
        ss = __fma_rn(w, w, ss);
      }
    }
    return warp_sum(ss);
  }
  __device__ __forceinline__ void norms(R sstep, R sdstep, double& z2, double& s2, double& x2) const {
    z2 = sumsq([&](R so, R, R xg) -> R { return softthres_fast(so - sstep * xg, sdstep); });
    s2 = sumsq([&](R so, R, R) -> R { return so; });
    x2 = sumsq([&](R, R, R xg) -> R { return xg; });
  }
  __device__ __forceinline__ double froot_sum(R sc, R sdc, R delta, double& dot) const {
    double s0 = 0.0, s1 = 0.0, d0 = 0.0, d1 = 0.0;
    for (long long i0 = b + lane; i0 < e; i0 += 128) {
      R so[4], xg[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const long long i = i0 + 32 * u;
        so[u] = i < e ? ysol[i] : R(0);  // zeros add nothing
        xg[u] = i < e ? xk[i] : R(0);
      }
      froot_term(so[0], xg[0], sc, sdc, delta, s0, d0);
      froot_term(so[1], xg[1], sc, sdc, delta, s1, d1);
      froot_term(so[2], xg[2], sc, sdc, delta, s0, d0);
      froot_term(so[3], xg[3], sc, sdc, delta, s1, d1);
    }
    dot = warp_sum(d0 + d1);
    return warp_sum(s0 + s1);
  }
};

template <class R> __device__ __forceinline__ bool adjacent_or_crossed(R a, R m, R b) { return !((a < m) && (m < b)); }

// x moved by k units in the last place (positive finite x)
__device__ __forceinline__ double ulp_step(double x, int k) {
  return __longlong_as_double(__double_as_longlong(x) + (long long)k);
}
__device__ __forceinline__ float ulp_step(float x, int k) { return __int_as_float(__float_as_int(x) + k); }

// Runs the bracket search of every group of the round in lockstep (lanes of one group hold identical
// copies of its state).  Returns the step c(n*) and whether the group's prox is zero.
//
// fzero(froot, lmin, lmax) (Roots' bisection) ends on two adjacent floats around the sign change of
// froot.  Same end state, an order of magnitude fewer evaluations: froot is smooth between the kinks of
// the soft threshold and nearly linear above the root, so safeguarded Newton steps from lmax (the
// derivative comes out of the same pass over the group) converge in three or four evaluations; as soon
// as a step lands within k ulps (k = 1, then 4, 16, ...) of an end of the bracket the next evaluation is placed k ulps inside
// that end -- stepping over the root, which leaves a bracket of k ulps that two or three midpoint steps
// close.  A step that leaves the bracket is replaced by the midpoint -- unless one end of the bracket already sits
// on the root, which is then stepped over -- and after 40 steps (never observed) the search degrades to plain
// bisection, which terminates by itself.
template <class R, class View>
__device__ __forceinline__ bool binf_solve(const View& gv, bool valid, R lam, R sigma, R delta, R& step_out) {
  const R eps = Eps<R>::value;
  const R sl = lam * sigma;  // σλ
  R dfx;                     // froot'(n) of the last evaluation
  auto froot = [&](R nn) -> R {  // :87-93
    const R gap = nn - sl;
    const R sc = div_fast(nn, gap);  // σ c(n)
    double dot;
    const double ss = gv.froot_sum(sc, delta * sc, delta, dot);
#ifdef SPX_GROUP_STATS
    if ((threadIdx.x & 31) == 0) atomicAdd(&g_stat_evals, 1ull);
#endif
    const R nw = (R)sqrt_fast(ss);
    // d‖w‖/dn = (w·dw/d(σc)) / ‖w‖ · d(σc)/dn,  d(σc)/dn = -σλ / (n - σλ)²
    dfx = R(1) + div_fast((R)dot * sl, nw * (gap * gap));
    return nn - nw;
  };
  const R lmin = sl * (R(1) + eps);
  const R ansatz = lmin + R(1);
  R step = ansatz / (sigma * (ansatz - sl));
  const R dstep = delta * step;
  // the three norms of :97-100 in one pass
  double z2 = 0.0, s2 = 0.0, x2 = 0.0;
  gv.norms(sigma * step, sigma * dstep, z2, s2, x2);
  const R zlmax = (R)sqrt_fast(z2) / sigma, nsol = (R)sqrt_fast(s2), nxk = (R)sqrt_fast(x2);
  const R lmax = nsol + sigma * (zlmax + R(1) * lam * nxk);  // |(ϵ-1)/ϵ + 1| = 1 for ϵ = 1  (:100)
  // One froot call site (the kernel is instruction-cache bound otherwise): trips 0 and 1 evaluate the two
  // ends of the bracket, the following ones are the search.
  R a = lmin, fa = R(0), bb = lmax, fb = R(0);
  R x = lmax, fx = R(0), dx = R(1);  // Newton state
  bool zero_out = false, done = !valid || !(lmin > R(0));
  int kulp = 1;
  for (int it = -2; it < 400; ++it) {
    R xn;
    bool probed = false;
    if (it < 0) {
      xn = (it == -2) ? lmin : lmax;
    } else {
      const R mid = a + (bb - a) / R(2);
      done = done || adjacent_or_crossed(a, mid, bb);
      if (!__any_sync(0xffffffffu, !done)) break;
      xn = mid;
      if (it < 40) {
        const R xs_ = x - div_fast(fx, dx);
        const bool inside = (a < xs_) && (xs_ < bb);
        if (inside) xn = xs_;
        // A Newton step that leaves the bracket while one end already sits on the root (|f| within 4096 ulps of n;
        // froot' >= 1: the norm it subtracts falls with n) -- Newton converged onto it from one side while the other
        // end is still far, the usual course when σλ >> ||sol|| (a sparse solution) and the root sits next to the
        // pole of c(n): step over that end instead of halving the distance to the far one ~50 times.  The vote keeps
        // this out of the common trip.
        if (__any_sync(0xffffffffu, !done && !inside)) {
          const R tiny = R(4096) * eps;
          if (!inside) xn = (jl_abs(fa) <= tiny * a) ? a : ((jl_abs(fb) <= tiny * bb) ? bb : mid);
        }
        const R a_k = ulp_step(a, kulp), b_k = ulp_step(bb, -kulp);
        if (xn <= a_k) {
          xn = (a_k < mid) ? a_k : mid;
          probed = true;
        } else if (xn >= b_k) {
          xn = (b_k > mid) ? b_k : mid;
          probed = true;
        }
      }
    }
    const R fn = froot(xn);
    if (it == -2) {
      fa = fn;
    } else if (it == -1) {
      fb = fn;
      fx = fn;
      dx = dfx;
      zero_out = fa * fb > R(0);
      done = done || zero_out || (fa != fa) || (fb != fb);
      if (!done && fa == R(0)) { bb = a; fb = R(0); done = true; }
      if (!done && fb == R(0)) { a = bb; fa = R(0); done = true; }
    } else if (!done) {
      x = xn;
      fx = fn;
      dx = dfx;
      if (fn == R(0)) {
        a = bb = xn;
        fa = fb = R(0);
        done = true;
      } else if ((fn < R(0)) == (fa < R(0))) {
        a = xn;
        fa = fn;
      } else {
        bb = xn;
        fb = fn;
      }
      if (probed) kulp = kulp < (1 << 20) ? kulp * 4 : kulp;
    }
  }
  if (!zero_out) {
    const R nroot = (jl_abs(fa) <= jl_abs(fb)) ? a : bb;
    step = nroot / (sigma * (nroot - sl));
    if (jl_abs(nroot - sl) == R(0)) zero_out = true;  // `abs(n - σλ) ≈ 0`  (:107)
  }
  step_out = step;
  return zero_out;
}

#ifndef SPX_GB_MINB
#define SPX_GB_MINB 3
#endif
template <class R, int PART>
__global__ void __launch_bounds__(kGroupThreads, PART == 0 ? SPX_GB_MINB : 2)
    group_l2binf_kernel(R* y, const R* xk, const R* sj, const R* q, long long ngroups,
                        const long long* __restrict__ offs, const R* __restrict__ lambda_g, R sigma, R delta,
                        UDiv<R> by_sigma, unsigned long long* task_counter, unsigned* long_flag,
                        const unsigned* __restrict__ uniform_flag, const unsigned char* __restrict__ done) {
  if (uniform_flag != nullptr && *uniform_flag != 0u) return;  // the uniform-layout kernels own this call
  if (PART == 1 && long_flag != nullptr && *long_flag == 0u) return;
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * kGroupThreads + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * kGroupThreads) >> 5;
  const long long ntasks = (ngroups + kTask - 1) / kTask;
  for (long long task = task_counter ? next_task(-1, 0, task_counter, lane) : warp; task < ntasks;
       task = next_task(task, nwarps, task_counter, lane)) {
    const long long g0 = task * kTask;
    const TaskHead th = load_task(offs, g0, ngroups, lane);
    // le[5]: groups of <= 256 elements (lanes beyond the task count as such)
    if (PART == 0 && th.le[5] != 0xffffffffu && long_flag != nullptr && lane == 0) *long_flag = 1u;
    if (PART == 1 ? (th.le[5] == 0xffffffffu) : (th.le[5] == 0u)) continue;
    const R lam_lane = lane < th.cnt ? lambda_g[g0 + lane] : R(0);
    int pos = 0;
    while (pos < th.cnt) {
      const int k = plan_round(th.le, pos);
      if (k < 0 && PART == 0) {
        if (long_flag != nullptr && lane == 0) *long_flag = 1u;
        pos += 1;
        continue;
      }
      if (k >= 0 && PART == 1) {
        pos += 32 >> k;
        continue;
      }
      if (k < 0) {  // long group: the whole warp, sol stashed in y
        if (done != nullptr && done[g0 + pos]) {  // solved by group_l2binf_big_kernel
          pos += 1;
          continue;
        }
        const long long b = __shfl_sync(0xffffffffu, th.lo, pos), e = __shfl_sync(0xffffffffu, th.hi, pos);
        const R lam = __shfl_sync(0xffffffffu, lam_lane, pos);
        for (long long i0 = b + lane; i0 < e; i0 += 128) {  // :80, loads batched (y may alias q)
          R s4[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const long long i = i0 + 32 * u;
            if (i < e) s4[u] = (ldv(q + i) + ldv(xk + i)) + ldv(sj + i);
          }
#pragma unroll
          for (int u = 0; u < 4; ++u)
            if (i0 + 32 * u < e) y[i0 + 32 * u] = s4[u];
        }
        LongView<R> gv{y, xk, b, e, lane, by_sigma};
        R step;
        const bool zero_out = binf_solve<R>(gv, true, lam, sigma, delta, step);
        const R sl = lam * sigma, dstep2 = delta * step;
        R alpha = R(0);
        if (!zero_out) {
          const double ss = gv.sumsq(
              [&](R so, R u, R xg) -> R { return so - sigma * softthres(u - step * xg, dstep2); });
          alpha = jl_max(R(0), R(1) - sl / (R)sqrt(ss));
        }
        for (long long i = b + lane; i < e; i += 32) {
          R o = R(0);
          const R so = y[i], xg = xk[i];
          if (!zero_out) o = alpha * (so - sigma * softthres(so / sigma - step * xg, dstep2));
          y[i] = o - (xg + sj[i]);
        }
#ifdef SPX_GROUP_STATS
        if (lane == 0) atomicAdd(&g_stat_groups, 1ull);
#endif
        pos += 1;
        continue;
      }
      if (done != nullptr) {  // groups the fast kernel has written: skip the round when none is left
        const int gi = pos + (lane >> k);
        const bool todo = gi < th.cnt && !done[g0 + gi];
        if (!__any_sync(0xffffffffu, todo)) {
          pos += 32 >> k;
          continue;
        }
      }
      Tile<R, false> t;
      t.load(th, k, pos, lane, xk, sj, q);
      if (done != nullptr && t.valid && done[g0 + t.group_in_task(pos, k, lane)]) {
        t.valid = false;  // already written: take part in the round's votes, store nothing
        t.e = t.b;
      }
      const R lam = __shfl_sync(0xffffffffu, lam_lane, t.group_in_task(pos, k, lane) & 31);
      TileView<R> gv{t, by_sigma};
      R step;
      const bool zero_out = binf_solve<R>(gv, t.valid, lam, sigma, delta, step);
      // y_g = l2prox(sol - σ softthres(sol/σ - step xk, Δ step), σλ) - (xk + sj)   (:109-116)
      const R sl = lam * sigma, dstep2 = delta * step;
      R w[kEPL];
      double ss = 0.0;
#pragma unroll
      for (int j = 0; j < kEPL; ++j) {
        w[j] = t.sol[j] - sigma * softthres_sel(by_sigma(t.sol[j]) - step * t.xkr[j], dstep2);
        ss += (double)w[j] * (double)w[j];
      }
      ss = sub_sum(ss, t.L);
      const R alpha = zero_out ? R(0) : jl_max(R(0), R(1) - sl / (R)sqrt_fast(ss));
#pragma unroll
      for (int j = 0; j < kEPL; ++j) {
        const long long i = t.b + (long long)j * t.L + t.sub;
        if (i < t.e) {
          const R o = zero_out ? R(0) : alpha * w[j];
          stv(y + i, o - (t.xkr[j] + sj[i]));
        }
      }
#ifdef SPX_GROUP_STATS
      if (t.valid && t.sub == 0) atomicAdd(&g_stat_groups, 1ull);
#endif
      pos += 32 >> k;
    }
  }
}

// ------------------------------------------- uniform layouts: the fast path --
// Every group has m = 8 L elements (L = 2, 4, ..., 32 lanes; m = 16 ... 256; C4 of BASELINE.json: m = 64) and
// the vector is 16-byte aligned.  No CSR planner, no per-element bounds tests: a warp round is 256 consecutive
// elements (32/L whole groups), each lane holds 8 elements of its group as 128-bit packets, offsets from the
// round base are compile-time constants.  spx_prox_groupl2binf_* takes this path when n == ngroups * m; a check
// kernel verifies offs[g] == g m on the device first (no host synchronisation: a flag gates either path).
//
// The root search (shiftedGroupNormL2Binf.jl:87-107).  froot(n) = n - ||w(τ)||, τ = σ c(n) = n/(n - σλ), with
// w_i = -τ (xk_i + Δ sign t_i) on the entries the soft threshold keeps and w_i = -sol_i on the others, i.e.
// ||w||² = τ² A + B, piecewise in τ; froot' >= 1, so the root is unique.
//   A  Float32 search (FP32 pipe, Float32 copies of sol and xk, Float32 sums): the three norms of :97-100, froot at
//      both ends of the bracket, then Newton on h(n) = (n - σλ) froot(n)/n -- linear in n when B = 0, where plain
//      Newton on froot crawls towards the pole of c(n) -- down to a step of 1e-5 n: three or four evaluations.
//      The signs of froot(lmin), froot(lmax) (`fl*fm > 0`, :102) are only taken from Float32 values 1e-4 away from 0.
//   B  one evaluation in R with Float64 sums; A and B of the current piece give froot', froot'' in closed form:
//      a Halley step lands on the root to ~1 ulp (cubic: 1e-6 -> 1e-18).
//   C  the final pass IS an evaluation: v = sol - σ softthres(sol/σ - c xk, Δc) = -w (:109), so ||v|| gives
//      froot(n) = n - ||v|| in the reference's own arithmetic.  |froot(n)| / froot'(n) <= max(2, min(16, 1/κ)) ulp(n),
//      κ = σλ/(n - σλ), accepts n (n is within that many ulps of the root, the distance bisection to
//      adjacent floats leaves between two summation orders).  Rounds that fail any check (NaN/Inf, magnitudes
//      outside the Float32 range, no clear sign, ill-conditioned roots next to the pole, residual not met) are
//      listed and redone by the bracketing search (binf_solve) in a second launch over the list.
template <class R> struct UVec {
  static constexpr int VEC = 16 / (int)sizeof(R);
  static constexpr int NCH = kEPL / VEC;
};
constexpr int kRoundElems = 32 * kEPL;  // 256 consecutive elements per warp round

// Each warp owns a private slice of shared memory -- planes q | xk | sj (even rounds) | sj (odd rounds), one round
// (256 elements) each -- that it fills with 16-byte cp.async copies one round AHEAD: while a round is being solved
// the next one is in flight, so the warp never waits on HBM between rounds (with three resident CTAs of eight
// warps, 144 KB per SM are in flight or staged).  A lane reads back exactly the 16-byte slots it copied itself:
// cp.async.wait_group is the only synchronisation.  sj has two planes because the current round still needs it
// for the store (y = ... - (xk + sj)) after the next round's copies have been issued.
template <class R, int L> struct UTile {
  R sol[kEPL], xkr[kEPL];
  int L_rt;  // == L (TileView reads a run-time width)
  bool valid;
  long long base;  // element index of the lane's first packet
  static constexpr int VEC = UVec<R>::VEC, NCH = UVec<R>::NCH;
  static constexpr uint32_t kPlane = kRoundElems * sizeof(R);  // bytes of one plane of one warp
  static constexpr uint32_t kWarpBytes = 4 * kPlane;
  static __device__ __forceinline__ bool lane_valid(long long round, long long ngroups, int lane) {
    return round * (32 / L) + lane / L < ngroups;
  }
  static __device__ __forceinline__ long long lane_base(long long round, int lane) {
    return round * kRoundElems + (long long)(lane / L) * (kEPL * L) + (lane % L) * VEC;
  }
  // enqueue the copies of `round` (every lane commits a group, possibly empty)
  static __device__ __forceinline__ void prefetch(long long round, long long ngroups, int lane, const R* xk, const R* sj,
                                                  const R* q, uint32_t sbase, int sjbuf) {
    if (lane_valid(round, ngroups, lane)) {
      const long long b = lane_base(round, lane);
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const uint32_t slot = sbase + (uint32_t)(c * 32 + lane) * 16u;
        cp_async16(slot, q + b + c * (L * VEC));
        cp_async16(slot + kPlane, xk + b + c * (L * VEC));
        cp_async16(slot + (2u + (uint32_t)sjbuf) * kPlane, sj + b + c * (L * VEC));
      }
    }
    cp_async_commit();
  }
  // the round whose copies were enqueued last.  STEP: the q plane holds ∇f, and q = (-ν) ∇f is formed here in R,
  // as spx_step_pre writes it
  template <bool STEP = false>
  __device__ __forceinline__ void take(long long round, long long ngroups, int lane, uint32_t sbase, int sjbuf,
                                       R mnu = R(0)) {
    cp_async_wait<0>();
    valid = lane_valid(round, ngroups, lane);
    base = lane_base(round, lane);
    L_rt = L;
    Pack<R, VEC> pq[NCH], px[NCH], ps[NCH];
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
#pragma unroll
      for (int e = 0; e < VEC; ++e) pq[c].v[e] = px[c].v[e] = ps[c].v[e] = R(0);
      if (valid) {
        const uint32_t slot = sbase + (uint32_t)(c * 32 + lane) * 16u;
        lds16(slot, pq[c]);
        lds16(slot + kPlane, px[c]);
        lds16(slot + (2u + (uint32_t)sjbuf) * kPlane, ps[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
      for (int e = 0; e < VEC; ++e) {
        if constexpr (STEP) pq[c].v[e] = mnu * pq[c].v[e];
        sol[c * VEC + e] = (pq[c].v[e] + px[c].v[e]) + ps[c].v[e];  // :80
        xkr[c * VEC + e] = px[c].v[e];
      }
  }
};
// TileView reads t.L
template <class R> struct UTileRef {
  const R (&sol)[kEPL];
  const R (&xkr)[kEPL];
  int L;
};

template <int L> __device__ __forceinline__ void usum2(float& a, float& b) {
#pragma unroll
  for (int o = L >> 1; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
}
template <int L> __device__ __forceinline__ void usum2(double& a, double& b) {
#pragma unroll
  for (int o = L >> 1; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
}
template <int L> __device__ __forceinline__ float usum(float a) {
#pragma unroll
  for (int o = L >> 1; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  return a;
}
template <int L> __device__ __forceinline__ double usum(double a) {
#pragma unroll
  for (int o = L >> 1; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  return a;
}

// ||w(τ)||² split into the thresholded entries (τ² A) and the others (B); T: arithmetic type, ACC: sum type
__device__ __forceinline__ float fma_t(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double fma_t(double a, double b, double c) { return __fma_rn(a, b, c); }
__device__ __forceinline__ float abs_t(float a) { return fabsf(a); }
__device__ __forceinline__ double abs_t(double a) { return fabs(a); }
__device__ __forceinline__ float cps_t(float a, float b) { return copysignf(a, b); }
__device__ __forceinline__ double cps_t(double a, double b) { return copysign(a, b); }
// accA += z² where the threshold keeps the entry (a > 0), accB += so² elsewhere: ONE predicated FMA each way (written
// in PTX: the compiler turns the C form into two FMAs and two selects).  A NaN excess counts as "not kept": it then
// poisons B through so or, for a finite so, is caught by the magnitude guards of the caller.
__device__ __forceinline__ void acc_pred(float a, float z, float so, float& accA, float& accB) {
  asm("{\n\t.reg .pred p;\n\tsetp.gt.f32 p, %2, 0f00000000;\n\t@p fma.rn.f32 %0, %3, %3, %0;\n\t@!p fma.rn.f32 %1, %4, %4, %1;\n\t}"
      : "+f"(accA), "+f"(accB)
      : "f"(a), "f"(z), "f"(so));
}
__device__ __forceinline__ void acc_pred(double a, double z, double so, double& accA, double& accB) {
  asm("{\n\t.reg .pred p;\n\tsetp.gt.f64 p, %2, 0d0000000000000000;\n\t@p fma.rn.f64 %0, %3, %3, %0;\n\t@!p fma.rn.f64 %1, %4, %4, %1;\n\t}"
      : "+d"(accA), "+d"(accB)
      : "d"(a), "d"(z), "d"(so));
}
__device__ __forceinline__ void acc_pred(float a, float z, float so, double& accA, double& accB) {
  acc_pred((double)a, (double)z, (double)so, accA, accB);
}
template <class T, class ACC>
__device__ __forceinline__ void binf_term(T so, T xg, T tau, T sdc, ACC& accA, ACC& accB) {
  const T t = fma_t(-tau, xg, so);
  const T a = abs_t(t) - sdc;
  const T z = cps_t(a, t) - so;
  acc_pred(a, z, so, accA, accB);
}
template <class T, class ACC, int L>
__device__ __forceinline__ void binf_eval(const T (&so)[kEPL], const T (&xg)[kEPL], T tau, T sdc, ACC& ssA, ACC& ssB) {
  ACC a0 = 0, a1 = 0, b0 = 0, b1 = 0;
#pragma unroll
  for (int j = 0; j < kEPL; j += 2) {
    binf_term<T, ACC>(so[j], xg[j], tau, sdc, a0, b0);
    binf_term<T, ACC>(so[j + 1], xg[j + 1], tau, sdc, a1, b1);
  }
  ssA = a0 + a1;
  ssB = b0 + b1;
  usum2<L>(ssA, ssB);
}

__device__ __forceinline__ float rcp_f(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// 1/x to ~1e-12 (the Halley correction needs no more)
__device__ __forceinline__ double rcp_d(double x) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  double e = __fma_rn(-x, y, 1.0);
  y = __fma_rn(y, e, y);
  e = __fma_rn(-x, y, 1.0);
  return __fma_rn(y, e, y);
}

// sol/σ for a warp-uniform σ without the out-of-range branch of div_uniform (callers guarantee normal operands;
// a zero numerator yields a zero of either sign, which the soft threshold maps to the same result)
__device__ __forceinline__ double quot_uniform(double a, const UDiv<double>& d) {
  const double q0 = a * d.y;
  const double r0 = __fma_rn(-d.s, q0, a);
  const double q1 = __fma_rn(r0, d.y, q0);
  const double r1 = __fma_rn(-d.s, q1, a);
  return __fma_rn(r1, d.y, q1);
}
__device__ __forceinline__ float quot_uniform(float a, const UDiv<float>& d) { return a / d.s; }

template <class R> struct LoCopy;
template <> struct LoCopy<double> {
  float so[kEPL], xg[kEPL];
  __device__ __forceinline__ void set(const double (&sol)[kEPL], const double (&xkr)[kEPL]) {
#pragma unroll
    for (int j = 0; j < kEPL; ++j) {
      so[j] = (float)sol[j];
      xg[j] = (float)xkr[j];
    }
  }
};

// The Float32 Newton search stops once a step is below this fraction of n: Newton converges quadratically, so the
// iterate that step leads to is already good to ~1e-6 n (Float32 noise level), and phase B cubes whatever is left
// (measured on the bench layouts: root within 3 ulps of the Float64 bisection either way, one evaluation fewer than
// with 1e-5).  A root phase B cannot repair fails the acceptance test and goes to the bracketing search.
constexpr float kBinfSearchTol = 2e-3f;
// Phases A and B.  Returns false when the round has to go through the bracketing search.  On success: zero_out
// (`fl*fm > 0`) and the root estimate n (R); fp_out = froot'(n).
template <class R, int L>
__device__ __forceinline__ bool binf_fast_search(const float (&so)[kEPL], const float (&xg)[kEPL],
                                                 const R (&sol)[kEPL], const R (&xkr)[kEPL], bool valid, R lam,
                                                 R sigma, R delta, R& n_out, double& fp_out, bool& zero_out) {
  const R epsR = Eps<R>::value;
  const R sl = lam * sigma;
  const R lmin = sl * (R(1) + epsR);
  const R ansatz = lmin + R(1);
  const R step_a = ansatz / (sigma * (ansatz - sl));
  const float slf = (float)sl, delf = (float)delta, lminf = (float)lmin;
  // ---- A: the three norms of :97-100 at τa = σ step(ansatz)
  const float tau_a = (float)sigma * (float)step_a;
  float z2 = 0.f, s2 = 0.f, x2 = 0.f, xmax = 0.f;
  {
    const float sdc = tau_a * delf;
#pragma unroll
    for (int j = 0; j < kEPL; ++j) {
      const float t = fmaf(-tau_a, xg[j], so[j]);
      const float a = fmaxf(fabsf(t) - sdc, 0.f);
      z2 = fmaf(a, a, z2);
      s2 = fmaf(so[j], so[j], s2);
      x2 = fmaf(xg[j], xg[j], x2);
      xmax = fmaxf(xmax, fabsf(xg[j]));
    }
    usum2<L>(z2, s2);
    x2 = usum<L>(x2);
#pragma unroll
    for (int o = L >> 1; o > 0; o >>= 1) xmax = fmaxf(xmax, __shfl_xor_sync(0xffffffffu, xmax, o));
  }
  const float nsolf = sqrt_approx(s2);
  const float lmaxf = nsolf + sqrt_approx(z2) + slf * sqrt_approx(x2);
  // magnitudes the Float32 search is trusted with (squares neither overflow nor flush; NaN fails every test)
  bool ok = (s2 > 1e-16f && s2 < 1e24f) && (x2 < 1e24f) && (z2 < 1e30f) && (delf < 1e12f) && (slf > 1e-12f && slf < 1e12f) &&
            (lmaxf > lminf * 1.001f);
  // ---- froot(lmin): τ = (1 + eps)/eps whatever σλ is.  An entry with |xk_i| clearly above Δ is thresholded there
  // and contributes τ (|xk_i| - Δ) -- orders of magnitude above lmin: froot(lmin) < 0 without evaluating it.
  const float tau_l = (float)((R(1) + epsR) / epsR);
  const float excess = xmax - delf;
  const bool fl_neg = (excess > 1e-4f * (xmax + delf)) && (excess * tau_l > 1e4f * (lminf + nsolf));
  float fl = -1.f;
  if (__any_sync(0xffffffffu, valid && ok && !fl_neg)) {
    float ssA, ssB;
    binf_eval<float, float, L>(so, xg, tau_l, tau_l * delf, ssA, ssB);
    const float nw = sqrt_approx(ssA + ssB);
    const float fle = lminf - nw;
    if (!fl_neg) {
      fl = fle;
      ok = ok && (fabsf(fl) > 1e-4f * fmaxf(lminf, nw));
    }
  }
  // ---- froot(lmax), then Newton on h(n) = (n - σλ) froot(n) / n
  float x = lmaxf, a_ = lminf, b_ = lmaxf;
  bool done = !valid || !ok;
  zero_out = false;
#pragma unroll 1
  for (int it = 0; it < 8; ++it) {
    const float gap = x - slf;
    const float rgap = rcp_f(gap), rx = rcp_f(x);
    const float tau = x * rgap;
    float ssA, ssB;
    binf_eval<float, float, L>(so, xg, tau, tau * delf, ssA, ssB);
    const float nw = sqrt_approx(ssA + ssB);
    const float fx = x - nw;
    // froot' = 1 + (Σ w dw/dτ) σλ / (||w|| gap²),  Σ w dw/dτ = τ A = ssA/τ
    const float dfx = fmaf(ssA * slf, rx * rcp_f(nw) * rgap, 1.f);
    if (it == 0) {
      ok = ok && (fabsf(fx) > 1e-4f * x);
      zero_out = (fl > 0.f) == (fx > 0.f);  // fl*fm > 0 (both are far from 0 here)
      done = done || !ok || zero_out;
    }
    // h = gap fx / x,  h' = (fx + gap (froot' - fx/x)) / x
    const float den = fmaf(gap, dfx - fx * rx, fx);
    const float stp = gap * fx * rcp_f(den);
    float xn = x - stp;
    const bool conv = (fabsf(stp) <= kBinfSearchTol * x) || (fx == 0.f);
    a_ = (fx < 0.f) ? x : a_;
    b_ = (fx < 0.f) ? b_ : x;
    if (!(xn >= a_ && xn <= b_)) xn = 0.5f * (a_ + b_);  // also catches NaN
    x = done ? x : xn;
    done = done || conv;
    if (!__any_sync(0xffffffffu, !done)) break;
  }
  ok = ok && done && (x == x);
  // ---- B: one evaluation in R with Float64 sums, Halley step
  const double xd = (double)x, sld = (double)sl;
  const double gapd = xd - sld;
  const double rg = rcp_d(gapd);
  const double taud = xd * rg;
  double ssA, ssB;
  binf_eval<R, double, L>(sol, xkr, (R)taud, (R)((double)delta * taud), ssA, ssB);
  const double ss = ssA + ssB;
  const double phi = sqrt_fast(ss);
  const double f = xd - phi;
  // φ = ||w||:  φ'τ' = -ssA σλ/(x φ gap),  φ''τ'² = ssA ssB σλ²/(x² φ³ gap²),  φ'τ'' = 2 ssA σλ/(x φ gap²)
  const double rD = rcp_d(xd * phi * gapd);
  const double p1 = ssA * sld * rD;  // -φ'τ'
  const double fp = 1.0 + p1;
  const double fpp = -(p1 * (ssB * sld * rD) * (rD * xd * gapd) + 2.0 * p1 * rg);
  const double n1 = xd - 2.0 * f * fp * rcp_d(__fma_rn(2.0 * fp, fp, -f * fpp));
  n_out = (R)n1;
  fp_out = fp;
  // ill-conditioned roots (next to the pole of c) and anything non-finite go to the bracketing search
  const double kap = sld * rcp_d(n1 - sld);
  ok = ok && (zero_out || (n1 > (double)lmin && kap < 64.0 && n1 == n1));
  return ok || !valid;
}
template <class R, int L>
__device__ __forceinline__ bool binf_fast_search_entry(const UTile<R, L>& t, R lam, R sigma, R delta, R& n_out,
                                                       double& fp_out, bool& zero_out);
template <int L>
__device__ __forceinline__ bool binf_fast_search_entry(const UTile<double, L>& t, double lam, double sigma, double delta,
                                                       double& n_out, double& fp_out, bool& zero_out) {
  LoCopy<double> lo;
  lo.set(t.sol, t.xkr);
  return binf_fast_search<double, L>(lo.so, lo.xg, t.sol, t.xkr, t.valid, lam, sigma, delta, n_out, fp_out, zero_out);
}
template <int L>
__device__ __forceinline__ bool binf_fast_search_entry(const UTile<float, L>& t, float lam, float sigma, float delta,
                                                       float& n_out, double& fp_out, bool& zero_out) {
  return binf_fast_search<float, L>(t.sol, t.xkr, t.sol, t.xkr, t.valid, lam, sigma, delta, n_out, fp_out, zero_out);
}

// the first round among i, i + stride, i + 2 stride, ... (below nrounds) that `declined` marks; nrounds when there is none
__device__ __forceinline__ long long first_declined(const unsigned char* declined, long long i, long long stride,
                                                    long long nrounds, int lane) {
  for (; i < nrounds; i += 32 * stride) {
    const long long r = i + lane * stride;
    const unsigned hit = __ballot_sync(0xffffffffu, r < nrounds && declined[r] != 0);
    if (hit != 0u) return i + (long long)(__ffs(hit) - 1) * stride;
  }
  return nrounds;
}

#ifndef SPX_GU_MINB
#define SPX_GU_MINB 3
#endif
// FAST: rounds grid-stride, failures appended to the work list.  !FAST: the listed rounds, bracketing search.
// STEP (spx_step_groupl2binf): y = s, q = ∇f; the store loop also writes xsy = (xk + sj) + s and sums ψ(s), Σ s² and
// Σ ∇f·s per CTA into part0[blockIdx.x] = {ψ, Σ s², infeasible} and part1[blockIdx.x] = {Σ ∇f·s, 0, redo}.  The FAST
// form also marks its declined rounds in `declined`, and the !FAST form walks those in round order on the same static
// round-to-warp map as the FAST one (not in the order of the work list, which is the order of atomicAdd), so that the
// sums come out the same on every call.  With the uniform flag at 0 both only raise `redo`.
// The Float64 STEP forms hold 8 more doubles per lane through the store loop and run with one CTA per SM fewer than
// the prox! forms (3 -> 2 and 2 -> 1), the occupancy at which they do not spill.
template <class R, int L, bool FAST, bool STEP = false>
__global__ void __launch_bounds__(kGroupThreads, (FAST ? SPX_GU_MINB : 2) - (STEP && sizeof(R) == 8 ? 1 : 0))
    group_l2binf_uniform_kernel(R* y, const R* xk, const R* sj, const R* q, long long ngroups,
                                const R* __restrict__ lambda_g, R sigma, R delta, UDiv<R> by_sigma,
                                const unsigned* __restrict__ uniform_flag, unsigned* wl_count, unsigned* wl_rounds,
                                R* xsy, R mnu, double rad, unsigned char* declined, Partial* part0, Partial* part1) {
  if (*uniform_flag == 0u) {
    if constexpr (STEP) {
      if (threadIdx.x == 0) {
        part0[blockIdx.x] = Partial{0.0, 0.0, -1};
        part1[blockIdx.x] = Partial{0.0, 0.0, 1};
      }
    }
    return;
  }
  constexpr int GPW = 32 / L;
  constexpr int VEC = UVec<R>::VEC, NCH = UVec<R>::NCH;
  constexpr bool SCAN = STEP && !FAST;  // walk the declined rounds of the static map
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * kGroupThreads + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * kGroupThreads) >> 5;
  const long long nrounds = FAST ? (ngroups + GPW - 1) / GPW
                            : SCAN ? (*wl_count == 0u ? 0 : (ngroups + GPW - 1) / GPW)
                                   : (long long)*wl_count;
  extern __shared__ __align__(16) unsigned char uni_smem[];
  const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(uni_smem) + (uint32_t)(threadIdx.x >> 5) * UTile<R, L>::kWarpBytes;
  auto round_of = [&](long long i) -> long long { return FAST || SCAN ? i : (long long)wl_rounds[i]; };
  // STEP: each thread's running ψ, Σ s² and Σ ∇f·s wait in shared memory between rounds, so that the search keeps
  // its registers
  __shared__ double uni_acc[STEP ? 3 : 1][STEP ? kGroupThreads : 1];
  if constexpr (STEP) uni_acc[0][threadIdx.x] = uni_acc[1][threadIdx.x] = uni_acc[2][threadIdx.x] = 0.0;
  bool infeasible = false;
  int sjbuf = 0;
  long long first = warp;
  if constexpr (SCAN) first = first_declined(declined, warp, nwarps, nrounds, lane);
  if (first < nrounds) UTile<R, L>::prefetch(round_of(first), ngroups, lane, xk, sj, q, sbase, 0);
  for (long long it = first; it < nrounds; it += nwarps, sjbuf ^= 1) {
    const long long round = round_of(it);
    if constexpr (SCAN) it = first_declined(declined, it + nwarps, nwarps, nrounds, lane) - nwarps;  // the next round taken is it + nwarps
    UTile<R, L> t;
    t.template take<STEP>(round, ngroups, lane, sbase, sjbuf, mnu);
    // the next round's copies go out now and land while this one is solved (q and xk planes are free again: their
    // contents sit in registers; sj goes to the other sj plane)
    if (it + nwarps < nrounds) UTile<R, L>::prefetch(round_of(it + nwarps), ngroups, lane, xk, sj, q, sbase, sjbuf ^ 1);
    const R lam = t.valid ? lambda_g[round * GPW + lane / L] : R(1);
    const R sl = lam * sigma;
    R nroot = R(0), step = R(0);
    double fp = 1.0;
    bool zero_out = false;
    if constexpr (FAST) {
      const bool ok = binf_fast_search_entry<L>(t, lam, sigma, delta, nroot, fp, zero_out);
      if (__any_sync(0xffffffffu, !ok)) {
        if (lane == 0) {
          wl_rounds[atomicAdd(wl_count, 1u)] = (unsigned)round;
          if constexpr (STEP) declined[round] = 1;
        }
        continue;
      }
    } else {
      UTileRef<R> ref{t.sol, t.xkr, L};
      TileView<R, UTileRef<R>> gv{ref, by_sigma};
      zero_out = binf_solve<R>(gv, t.valid, lam, sigma, delta, step);
    }
    // ---- C: y_g = l2prox(sol - σ softthres(sol/σ - step xk, Δ step), σλ) - (xk + sj)   (:109-116)
    R w[kEPL];
    // the fast rounds hold magnitudes far inside the normal range (guards of binf_fast_search): their scalar
    // quotients take the branch-free ~1 ulp division, their sol/σ the correctly rounded quotient without its
    // out-of-range test
    if (FAST) step = div_fast(nroot, sigma * (nroot - sl));  // c(n)  (:85)
    const R dstep2 = delta * step;
    double ss = 0.0;
#pragma unroll
    for (int j = 0; j < kEPL; ++j) {
      const R u = FAST ? quot_uniform(t.sol[j], by_sigma) : by_sigma(t.sol[j]);
      w[j] = t.sol[j] - sigma * softthres_sel(u - step * t.xkr[j], dstep2);
      ss = __fma_rn((double)w[j], (double)w[j], ss);
    }
    ss = usum<L>(ss);
    const R nv = (R)sqrt_fast(ss);
    const R alpha = zero_out ? R(0) : jl_max(R(0), R(1) - (FAST ? div_fast(sl, nv) : sl / nv));
    if (FAST) {
      // froot(nroot) = nroot - ||v|| in the reference's arithmetic: the acceptance test of the fast search
      const R res = nroot - nv;
      const R gap = nroot - sl;
      // n is within |res| / froot'(n) of the root (froot' >= 1, ~1 + κ next to the pole -- where the residual's own
      // rounding noise grows with κ as well): accepted within max(2, min(16, 1/κ)) ulps of the ROOT, κ = σλ/gap
      const R ulps = jl_max(R(2), jl_min(R(16), gap * (R)(1.0 / (double)sl)));
      const bool accepted = zero_out || !t.valid || (jl_abs(res) <= ulps * Eps<R>::value * nroot * (R)fp);
      if (__any_sync(0xffffffffu, !accepted)) {
        if (lane == 0) {
          wl_rounds[atomicAdd(wl_count, 1u)] = (unsigned)round;
          if constexpr (STEP) declined[round] = 1;
        }
        continue;
      }
    }
    if constexpr (STEP) {
      // ∇f of this round again for Σ ∇f·s: its q plane already holds the next round, and the copy of one round
      // ago left it in L2
      double vv = 0.0, ss2 = 0.0, dot = 0.0;
      if (t.valid) {
        Pack<R, VEC> pg[NCH];
#pragma unroll
        for (int c = 0; c < NCH; ++c) ld_stream(q + t.base + c * (L * VEC), pg[c]);
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          Pack<R, VEC> ps, po, px;
          lds16(sbase + (2u + (uint32_t)sjbuf) * UTile<R, L>::kPlane + (uint32_t)(c * 32 + lane) * 16u, ps);
#pragma unroll
          for (int e = 0; e < VEC; ++e) {
            const int j = c * VEC + e;
            const R o = zero_out ? R(0) : alpha * w[j];
            const R xs = t.xkr[j] + ps.v[e];
            po.v[e] = o - xs;
            px.v[e] = xs + po.v[e];  // the generic ψ argument (xk + sj) + s
            // ψ(s) in the association of group_value_kernel: w = sj + s against the ball, v = w + xk
            const R wv = ps.v[e] + po.v[e];
            infeasible = infeasible || (double)wv < -rad || (double)wv > rad;
            const R v = wv + t.xkr[j];
            vv += (double)v * (double)v;
            ss2 = __fma_rn((double)po.v[e], (double)po.v[e], ss2);
            dot = __fma_rn((double)pg[c].v[e], (double)po.v[e], dot);
          }
          st_stream(y + t.base + c * (L * VEC), po);
          if (xsy != nullptr) st_stream(xsy + t.base + c * (L * VEC), px);
        }
      }
      vv = usum<L>(vv);
      if (t.valid && lane % L == 0) uni_acc[0][threadIdx.x] += (double)(lam * (R)sqrt_fast(vv));  // λ_g ‖v_g‖  groupNormL2.jl:36
      uni_acc[1][threadIdx.x] += ss2;
      uni_acc[2][threadIdx.x] += dot;
    } else if (t.valid) {
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        Pack<R, VEC> ps, po;
        lds16(sbase + (2u + (uint32_t)sjbuf) * UTile<R, L>::kPlane + (uint32_t)(c * 32 + lane) * 16u, ps);
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
          const int j = c * VEC + e;
          const R o = zero_out ? R(0) : alpha * w[j];
          po.v[e] = o - (t.xkr[j] + ps.v[e]);
        }
        st_stream(y + t.base + c * (L * VEC), po);
      }
    }
  }
  if constexpr (STEP) {
    Partial p{uni_acc[0][threadIdx.x], uni_acc[1][threadIdx.x], infeasible ? 1 : -1};
    p = block_fold<kGroupThreads>(p);
    Partial p2{uni_acc[2][threadIdx.x], 0.0, -1};
    p2 = block_fold<kGroupThreads>(p2);
    if (threadIdx.x == 0) {
      part0[blockIdx.x] = p;
      part1[blockIdx.x] = p2;
    }
  }
}

// ---- ragged groups of <= 256 elements: the fast search on the warp rounds of the CSR planner ------------------------
// Same rounds as group_l2binf_kernel<R, 0> (32 >> k groups of 1 << k lanes, 8 zero-padded elements per lane), same
// search and acceptance test as the uniform-layout kernel, but per GROUP: an accepted group is written and marked in
// `done`, anything else is left to the bracketing search that runs afterwards.
template <class R, int L>
__device__ __forceinline__ bool binf_tile_search(const Tile<R, true>& t, R lam, R sigma, R delta, R& nroot, double& fp,
                                                 bool& zero_out) {
  if constexpr (sizeof(R) == 8) {
    LoCopy<double> lo;
    lo.set(t.sol, t.xkr);
    return binf_fast_search<double, L>(lo.so, lo.xg, t.sol, t.xkr, t.valid, lam, sigma, delta, nroot, fp, zero_out);
  } else {
    return binf_fast_search<float, L>(t.sol, t.xkr, t.sol, t.xkr, t.valid, lam, sigma, delta, nroot, fp, zero_out);
  }
}

template <class R>
__global__ void __launch_bounds__(kGroupThreads, sizeof(R) == 8 ? 2 : 3)
    group_l2binf_small_fast_kernel(R* y, const R* xk, const R* sj, const R* q, long long ngroups,
                                   const long long* __restrict__ offs, const R* __restrict__ lambda_g, R sigma, R delta,
                                   UDiv<R> by_sigma, const unsigned* __restrict__ uniform_flag,
                                   unsigned char* __restrict__ done) {
  if (uniform_flag != nullptr && *uniform_flag != 0u) return;
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * kGroupThreads + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * kGroupThreads) >> 5;
  const long long ntasks = (ngroups + kTask - 1) / kTask;
  for (long long task = warp; task < ntasks; task += nwarps) {
    const long long g0 = task * kTask;
    const TaskHead th = load_task(offs, g0, ngroups, lane);
    if (th.le[5] == 0u) continue;  // no group of <= 256 elements in this task
    const R lam_lane = lane < th.cnt ? lambda_g[g0 + lane] : R(0);
    int pos = 0;
    while (pos < th.cnt) {
      const int k = plan_round(th.le, pos);
      if (k < 0) {
        pos += 1;
        continue;
      }
      Tile<R, true> t;
      t.load(th, k, pos, lane, xk, sj, q);
      const int gi = t.group_in_task(pos, k, lane);
      const R lam = __shfl_sync(0xffffffffu, lam_lane, gi & 31);
      const R sl = lam * sigma;
      R nroot = R(0);
      double fp = 1.0;
      bool zero_out = false, ok = false;
      switch (k) {
        case 0: ok = binf_tile_search<R, 1>(t, lam, sigma, delta, nroot, fp, zero_out); break;
        case 1: ok = binf_tile_search<R, 2>(t, lam, sigma, delta, nroot, fp, zero_out); break;
        case 2: ok = binf_tile_search<R, 4>(t, lam, sigma, delta, nroot, fp, zero_out); break;
        case 3: ok = binf_tile_search<R, 8>(t, lam, sigma, delta, nroot, fp, zero_out); break;
        case 4: ok = binf_tile_search<R, 16>(t, lam, sigma, delta, nroot, fp, zero_out); break;
        default: ok = binf_tile_search<R, 32>(t, lam, sigma, delta, nroot, fp, zero_out); break;
      }
      // y_g = l2prox(sol - σ softthres(sol/σ - step xk, Δ step), σλ) - (xk + sj)   (:109-116) and the acceptance test
      const R step = div_fast(nroot, sigma * (nroot - sl));  // c(n)  (:85)
      const R dstep2 = delta * step;
      R w[kEPL];
      double ss = 0.0;
#pragma unroll
      for (int j = 0; j < kEPL; ++j) {
        w[j] = t.sol[j] - sigma * softthres_sel(quot_uniform(t.sol[j], by_sigma) - step * t.xkr[j], dstep2);
        ss = __fma_rn((double)w[j], (double)w[j], ss);
      }
      ss = sub_sum(ss, t.L);
      const R nv = (R)sqrt_fast(ss);
      const R res = nroot - nv;
      const R gap = nroot - sl;
      const R ulps = jl_max(R(2), jl_min(R(16), gap * (R)(1.0 / (double)sl)));
      const bool accepted = ok && (zero_out || (jl_abs(res) <= ulps * Eps<R>::value * nroot * (R)fp));
      if (t.valid && accepted) {
        const R alpha = zero_out ? R(0) : jl_max(R(0), R(1) - div_fast(sl, nv));
#pragma unroll
        for (int j = 0; j < kEPL; ++j) {
          const long long i = t.b + (long long)j * t.L + t.sub;
          if (i < t.e) stv(y + i, (zero_out ? R(0) : alpha * w[j]) - t.xs[j]);
        }
        if (t.sub == 0) done[g0 + gi] = 1;
      }
      pos += 32 >> k;
    }
  }
}

// ---- one CTA per group of 1025..4096 elements (ShiftedGroupNormL2Binf) ----------------------------------------------
// The warp path above keeps a long group in the output vector and re-reads it from L2 for every evaluation of froot:
// with groups of thousands of elements nearly all of a ragged vector goes through one warp per group.  Here the group
// sits in the shared memory of a 256-thread CTA in R (sol | xk | sj, 8 or 16 elements per thread; q | xk | sj arrive by
// three bulk copies of one elected thread, as in group_l2_big_kernel: no per-element copy instructions) with Float32 copies
// of sol and xk in registers; every evaluation of the search is a pass over those registers plus one block reduction
// (a single __syncthreads: the reduction slots alternate).  The search is the one of the uniform path: froot(lmin)
// skipped when its sign is certain, Newton on h(n) = (n - σλ) froot(n)/n from lmax in Float32, one evaluation in R with
// Float64 sums and a Halley step, then the final pass as the acceptance test (|froot(n)| / froot'(n) within
// max(2, min(16, 1/κ)) ulps of n).  Groups that fail a guard or the test are left -- unmarked in `done` -- to the
// bracketing search of the warp path, which runs afterwards.  (The all-R search this replaces spent 293 thread
// instructions per element, most of them Float64, on the ragged layout.)
constexpr int kBinfBigThreads = 256;  // two CTAs per SM, 16 (or 8) elements per thread; 512 threads x 8 measured slower
constexpr int kBinfMidThreads = 128;  // groups of 257..512 and 513..1024 elements: eight CTAs per SM, 4 and 8 elements per thread
template <int T> struct BigRed {
  double v[2][T / 32][4];
};
// sums a[0..N) over the CTA; every thread gets the totals.  One barrier per call (slots alternate by `parity`).
template <int N, int T> __device__ __forceinline__ void block_sums(double (&a)[N], BigRed<T>& red, int& parity) {
#pragma unroll
  for (int k = 0; k < N; ++k) a[k] = warp_sum(a[k]);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < N; ++k) red.v[parity][w][k] = a[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < N; ++k) {
    double t = 0.0;
#pragma unroll
    for (int ww = 0; ww < T / 32; ++ww) t += red.v[parity][ww][k];
    a[k] = t;
  }
  parity ^= 1;
}

template <int T> struct BigRedF {
  float v[2][T / 32][4];
};
// Float32 form for the search: sums a[0..N) (N <= 3) and, when mx is given, the maximum of *mx over the CTA
template <int N, int T>
__device__ __forceinline__ void block_sums_f(float (&a)[N], BigRedF<T>& red, int& parity, float* mx = nullptr) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int k = 0; k < N; ++k) a[k] += __shfl_xor_sync(0xffffffffu, a[k], o);
    if (mx) *mx = fmaxf(*mx, __shfl_xor_sync(0xffffffffu, *mx, o));
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < N; ++k) red.v[parity][w][k] = a[k];
    if (mx) red.v[parity][w][3] = *mx;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < N; ++k) {
    float t = 0.f;
#pragma unroll
    for (int ww = 0; ww < T / 32; ++ww) t += red.v[parity][ww][k];
    a[k] = t;
  }
  if (mx) {
    float m = 0.f;
#pragma unroll
    for (int ww = 0; ww < T / 32; ++ww) m = fmaxf(m, red.v[parity][ww][3]);
    *mx = m;
  }
  parity ^= 1;
}

// one group, E elements per thread (E T >= m).  Returns true when y_g has been written.
// The search runs on Float32 copies of sol and xk held in registers (Float32 sums, one barrier per evaluation); the
// group itself stays in the staging planes in R -- sol (later w) | xk | sj, every thread reading and writing only its
// own slots -- for the one evaluation in R with Float64 sums (Halley step) and the final pass, which is the acceptance
// test.  What the search did therefore cannot reach y except through a root the final pass has accepted.
// q | xk | sj of the group arrive in the planes (PLS elements each: bulk_plane) by three bulk copies issued by thread 0
// once every thread is done with the previous group (the barrier below), completion on `bar`.
template <class R, int E, int T, int PLS>
__device__ __forceinline__ bool binf_big_group(R* y, const R* xk, const R* sj, const R* q, long long b, long long e,
                                               R lam, R sigma, R delta, const UDiv<R>& by_sigma, BigRed<T>& red,
                                               BigRedF<T>& redf, int& parity, int& parity_f, R* stage, uint64_t* bar,
                                               uint32_t& phase) {
  const int t = threadIdx.x;
  const R epsR = Eps<R>::value;
  const R sl = lam * sigma;
  float so[E], xg[E];
  // slots in use: ne per thread (CTA-uniform; the loops below skip the others), element k T + t of the group in slot k
  const int m = (int)(e - b), ne = (m + T - 1) / T;
  __syncthreads();  // the planes are free: every thread has finished the previous group
  if (t == 0) {
    fence_proxy_async();
    stage_group_bulk<R, 3, PLS>(stage, bar, q, xk, sj, b, e);
  }
  // each thread works on its own slots from here on (element k T + t of the group; the planes carry the padding of
  // the 16-byte granule the group starts in)
  R* const st_q = stage + bulk_skip(q + b) + t;
  R* const st_x = stage + PLS + bulk_skip(xk + b) + t;
  R* const st_s = stage + 2 * PLS + bulk_skip(sj + b) + t;
  mbar_wait(bar, phase);
  phase ^= 1u;
  // sol over q in the plane; slots beyond the group hold zeros (they add nothing to any sum below)
#pragma unroll
  for (int k = 0; k < E; ++k) {
    const int i = k * T + t;
    R s = R(0), xi = R(0);
    if (i < m) {
      xi = st_x[k * T];
      s = (st_q[k * T] + xi) + st_s[k * T];  // :80
    } else {
      st_x[k * T] = R(0);
    }
    st_q[k * T] = s;
    so[k] = (float)s;
    xg[k] = (float)xi;
  }
  // ---- A: the three norms of :97-100 (and max |xk|) at τa = σ c(lmin + 1), in Float32
  const R lmin = sl * (R(1) + epsR);
  const R ansatz = lmin + R(1);
  const R step_a = ansatz / (sigma * (ansatz - sl));
  const float slf = (float)sl, delf = (float)delta, lminf = (float)lmin;
  const float tau_a = (float)sigma * (float)step_a;
  float nm[3] = {0.f, 0.f, 0.f}, xmax = 0.f;
  {
    const float sdc = tau_a * delf;
#pragma unroll
    for (int k = 0; k < E; ++k) {
      if (k >= ne) break;
      const float tt = fmaf(-tau_a, xg[k], so[k]);
      const float a = fmaxf(fabsf(tt) - sdc, 0.f);
      nm[0] = fmaf(a, a, nm[0]);
      nm[1] = fmaf(so[k], so[k], nm[1]);
      nm[2] = fmaf(xg[k], xg[k], nm[2]);
      xmax = fmaxf(xmax, fabsf(xg[k]));
    }
    block_sums_f<3, T>(nm, redf, parity_f, &xmax);
  }
  const float nsolf = sqrt_approx(nm[1]);
  const float lmaxf = nsolf + sqrt_approx(nm[0]) + slf * sqrt_approx(nm[2]);
  // magnitudes the Float32 search is trusted with (see binf_fast_search); everything else: the bracketing search
  bool ok = (nm[1] > 1e-16f && nm[1] < 1e24f) && (nm[2] < 1e24f) && (nm[0] < 1e30f) && (delf < 1e12f) &&
            (slf > 1e-12f && slf < 1e12f) && (lmaxf > lminf * 1.001f);
  auto eval = [&](float tau, float& ssA, float& ssB) {
    float a0 = 0.f, a1 = 0.f, b0 = 0.f, b1 = 0.f;
    const float sdc = tau * delf;
#pragma unroll
    for (int k = 0; k < E; k += 2) {
      if (k >= ne) break;
      binf_term<float, float>(so[k], xg[k], tau, sdc, a0, b0);
      binf_term<float, float>(so[k + 1], xg[k + 1], tau, sdc, a1, b1);
    }
    float ab[2] = {a0 + a1, b0 + b1};
#ifdef SPX_GROUP_STATS
    if (threadIdx.x == 0) atomicAdd(&g_stat_big[0], 1ull);
#endif
    block_sums_f<2, T>(ab, redf, parity_f);
    ssA = ab[0];
    ssB = ab[1];
  };
  // froot(lmin) < 0 for certain when some |xk_i| is clearly above Δ (see binf_fast_search)
  const float tau_l = (float)((R(1) + epsR) / epsR);
  const float excess = xmax - delf;
  const bool fl_neg = (excess > 1e-4f * (xmax + delf)) && (excess * tau_l > 1e4f * (lminf + nsolf));
  float fl = -1.f;
  if (ok && !fl_neg) {  // CTA-uniform: every thread holds the same scalars
    float ssA, ssB;
    eval(tau_l, ssA, ssB);
    const float nw = sqrt_approx(ssA + ssB);
    fl = lminf - nw;
    ok = ok && (fabsf(fl) > 1e-4f * fmaxf(lminf, nw));
  }
  // froot(lmax), then Newton on h(n) = (n - σλ) froot(n)/n
  float x = lmaxf, a_ = lminf, b_ = lmaxf;
  bool zero_out = false, conv = false;
  if (ok) {
#pragma unroll 1
    for (int it = 0; it < 8; ++it) {
      const float gap = x - slf;
      const float rgap = rcp_f(gap), rx = rcp_f(x);
      const float tau = x * rgap;
      float ssA, ssB;
      eval(tau, ssA, ssB);
      const float nw = sqrt_approx(ssA + ssB);
      const float fx = x - nw;
      const float dfx = fmaf(ssA * slf, rx * rcp_f(nw) * rgap, 1.f);  // froot' = 1 + (ssA/τ) σλ / (||w|| gap²)
      if (it == 0) {
        ok = fabsf(fx) > 1e-4f * x;
        zero_out = (fl > 0.f) == (fx > 0.f);  // fl*fm > 0  (:102)
        if (!ok || zero_out) break;
      }
      const float den = fmaf(gap, dfx - fx * rx, fx);
      const float stp = gap * fx * rcp_f(den);
      float xn = x - stp;
      conv = (fabsf(stp) <= kBinfSearchTol * x) || (fx == 0.f);
      a_ = (fx < 0.f) ? x : a_;
      b_ = (fx < 0.f) ? b_ : x;
      if (!(xn >= a_ && xn <= b_)) xn = 0.5f * (a_ + b_);  // also catches NaN
      x = xn;
      if (conv) break;
    }
  }
  ok = ok && (zero_out || conv) && (x == x);
  if (!ok) return false;
  R nroot = R(0);
  double fp = 1.0;
  if (!zero_out) {
    // ---- B: one evaluation in R with Float64 sums at the Float32 root, Halley step (as in binf_fast_search)
    const double xd = (double)x, sld = (double)sl;
    const double gapd = xd - sld;
    const double rg = rcp_d(gapd);
    const double taud = xd * rg;
    double ab[2];
    {
      const R tau = (R)taud, sdc = (R)((double)delta * taud);
      double a0 = 0.0, a1 = 0.0, b0 = 0.0, b1 = 0.0;
#pragma unroll
      for (int k = 0; k < E; k += 2) {
        if (k >= ne) break;
        binf_term<R, double>(st_q[k * T], st_x[k * T], tau, sdc, a0, b0);
        binf_term<R, double>(st_q[(k + 1) * T], st_x[(k + 1) * T], tau, sdc, a1, b1);
      }
      ab[0] = a0 + a1;
      ab[1] = b0 + b1;
#ifdef SPX_GROUP_STATS
      if (threadIdx.x == 0) atomicAdd(&g_stat_big[0], 1ull);
#endif
      block_sums<2, T>(ab, red, parity);
    }
    const double ssA = ab[0], ssB = ab[1];
    const double phi = sqrt_fast(ssA + ssB);
    const double f = xd - phi;
    const double rD = rcp_d(xd * phi * gapd);
    const double p1 = ssA * sld * rD;
    fp = 1.0 + p1;
    const double fpp = -(p1 * (ssB * sld * rD) * (rD * xd * gapd) + 2.0 * p1 * rg);
    const double n1 = xd - 2.0 * f * fp * rcp_d(__fma_rn(2.0 * fp, fp, -f * fpp));
    nroot = (R)n1;
    const double kap = sld * rcp_d(n1 - sld);
    if (!(n1 > (double)lmin && kap < 64.0 && n1 == n1)) return false;  // next to the pole of c, or not finite
  }
  // ---- y_g = l2prox(sol - σ softthres(sol/σ - c xk, Δ c), σλ) - (xk + sj)   (:109-116), and the acceptance test
  R alpha = R(0);
  if (!zero_out) {
    const R step = div_fast(nroot, sigma * (nroot - sl));
    const R dstep2 = delta * step;
    double vs[1] = {0.0};
#pragma unroll
    for (int k = 0; k < E; ++k) {  // w overwrites sol
      if (k >= ne) break;
      const R s = st_q[k * T];
      const R w = s - sigma * softthres_sel(quot_uniform(s, by_sigma) - step * st_x[k * T], dstep2);
      st_q[k * T] = w;
      vs[0] = __fma_rn((double)w, (double)w, vs[0]);
    }
    block_sums<1, T>(vs, red, parity);
    const R nv = (R)sqrt_fast(vs[0]);
    const R res = nroot - nv;
    const R gap = nroot - sl;
    // within max(2, min(16, 1/κ)) ulps of the root: |res| / froot' (see group_l2binf_uniform_kernel)
    const R ulps = jl_max(R(2), jl_min(R(16), gap * (R)(1.0 / (double)sl)));
    if (!(jl_abs(res) <= ulps * epsR * nroot * (R)fp)) return false;  // not accepted: the bracketing search takes it
    alpha = jl_max(R(0), R(1) - div_fast(sl, nv));
  }
  R* const gy = y + b;
#pragma unroll
  for (int k = 0; k < E; ++k) {
    const int i = k * T + t;
    if (k < ne && i < m) {
      const R o = zero_out ? R(0) : alpha * st_q[k * T];
      stv(gy + i, o - (st_x[k * T] + st_s[k * T]));
    }
  }
  return true;
}

// T threads per group; groups of LO < m <= EA T elements with EA elements per thread, up to EB T with EB
// TPS: threads per SM the register budget is set for (512: 128 registers, 1024: 64)
template <class R, int T, int LO, int EA, int EB, int TPS>
__global__ void __launch_bounds__(T, TPS / T)
    group_l2binf_big_kernel(R* y, const R* xk, const R* sj, const R* q, long long ngroups,
                            const long long* __restrict__ offs, const R* __restrict__ lambda_g, R sigma, R delta,
                            UDiv<R> by_sigma, const unsigned* __restrict__ uniform_flag, unsigned char* __restrict__ done) {
  if (uniform_flag != nullptr && *uniform_flag != 0u) return;
  constexpr int PL = EB * T;                 // longest group of the class
  constexpr int PLS = bulk_plane<R>(PL);     // elements per staging plane
  __shared__ int list[T];
  __shared__ int wcount[T / 32];
  __shared__ BigRed<T> red;
  __shared__ BigRedF<T> redf;
  __shared__ __align__(8) uint64_t bar;
  extern __shared__ __align__(128) unsigned char big_stage_raw[];
  R* const stage = reinterpret_cast<R*>(big_stage_raw);  // three planes of PLS elements: q | xk | sj
  // No StageRing here: the stage is the group's working memory (sol, then w) until the final pass, so it cannot take
  // the next group early, and only one stage of 3 x 4096 elements fits per CTA.  The next group goes to L2 instead.
  const int t = threadIdx.x;
  if (t == 0) mbar_init(&bar, 1);
  __syncthreads();
  uint32_t phase = 0;
  int parity = 0, parity_f = 0;
  for (long long g0 = (long long)blockIdx.x * T; g0 < ngroups; g0 += (long long)gridDim.x * T) {
    const int nbig = list_class_groups<T, LO, PL>(offs, g0, ngroups, list, wcount);
    for (int j = 0; j < nbig; ++j) {
      const long long g = g0 + list[j];
      const long long b = offs[g], e = offs[g + 1];
      const R lam = lambda_g[g];
      if (j + 1 < nbig) {
        const long long gn = g0 + list[j + 1];
        prefetch_group_l2<R, T>(q, xk, sj, offs[gn], offs[gn + 1]);
      }
      bool wrote;
      if (e - b <= EA * T)
        wrote = binf_big_group<R, EA, T, PLS>(y, xk, sj, q, b, e, lam, sigma, delta, by_sigma, red, redf, parity, parity_f, stage, &bar, phase);
      else
        wrote = binf_big_group<R, EB, T, PLS>(y, xk, sj, q, b, e, lam, sigma, delta, by_sigma, red, redf, parity, parity_f, stage, &bar, phase);
      if (wrote && t == 0) done[g] = 1;
#ifdef SPX_GROUP_STATS
      if (t == 0) atomicAdd(&g_stat_big[wrote ? 1 : 2], 1ull);
#endif
    }
  }
}

// flag = 1 iff offs[g] == g m for every g <= ngroups (grid-stride; the flag starts at 1)
__global__ void __launch_bounds__(256) group_uniform_check_kernel(const long long* __restrict__ offs, long long ngroups,
                                                                  long long m, unsigned* flag) {
  bool bad = false;
  for (long long g = (long long)blockIdx.x * 256 + threadIdx.x; g <= ngroups; g += (long long)gridDim.x * 256)
    bad = bad || (offs[g] != g * m);
  if (__syncthreads_or(bad) && threadIdx.x == 0) *flag = 0u;
}

// ----------------------------------------------------- group values (ψ(y)) --
// ShiftedGroupNormL2: v = (xk + sj) + y  (ShiftedProximalOperators.jl:51-54)
// ShiftedGroupNormL2Binf: w = sj + y, IndBallLinf(1.1Δ)(w), v = w + xk
// (shiftedGroupNormL2Binf.jl:34-39); value Σ_g λ_g ‖v_g‖  (groupNormL2.jl:33-39)
template <class R, int PART>
__global__ void __launch_bounds__(kGroupThreads)
    group_value_kernel(const R* __restrict__ xk, const R* __restrict__ sj, const R* __restrict__ y, long long ngroups,
                       const long long* __restrict__ offs, const R* __restrict__ lambda_g, bool binf, double rad,
                       unsigned classes, Partial* __restrict__ partials) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * kGroupThreads + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * kGroupThreads) >> 5;
  const long long ntasks = (ngroups + kTask - 1) / kTask;
  Partial p;
  p.s = 0.0;
  p.s2 = 0.0;
  p.bad = -1;
  // v = (xk + sj) + y, or for the Binf form w = sj + y (checked against the ball) and v = w + xk
  auto term = [&](R xi, R si, R yi) -> double {
    R v;
    if (binf) {
      const R w = si + yi;
      if ((double)w < -rad || (double)w > rad) p.bad = 1;
      v = w + xi;
    } else {
      v = (xi + si) + yi;
    }
    return (double)v * (double)v;
  };
  for (long long task = warp; task < ntasks; task += nwarps) {
    const long long g0 = task * kTask;
    const TaskHead th = load_task(offs, g0, ngroups, lane);
    // le[5]: groups of <= 256 elements (lanes beyond the task count as such)
    if (PART == 1 ? (th.le[5] == 0xffffffffu) : (th.le[5] == 0u)) continue;
    const R lam_lane = lane < th.cnt ? lambda_g[g0 + lane] : R(0);
    int pos = 0;
    while (pos < th.cnt) {
      const int k = plan_round(th.le, pos);
      if (k < 0) {  // long group: the whole warp
        const long long b = __shfl_sync(0xffffffffu, th.lo, pos), e = __shfl_sync(0xffffffffu, th.hi, pos);
        if (PART == 1 && !in_launched_class(e - b, classes)) {
          double ss = 0.0;
#pragma unroll 4
          for (long long i = b + lane; i < e; i += 32) ss += term(xk[i], sj[i], y[i]);
          ss = warp_sum(ss);
          const R lam = __shfl_sync(0xffffffffu, lam_lane, pos);
          if (lane == 0) p.s += (double)(lam * (R)sqrt(ss));
        }
        pos += 1;
        continue;
      }
      if (PART == 1) {
        pos += 32 >> k;
        continue;
      }
      const int L = 1 << k, sub = lane & (L - 1), gi = pos + (lane >> k);
      const long long lo = __shfl_sync(0xffffffffu, th.lo, gi & 31), hi = __shfl_sync(0xffffffffu, th.hi, gi & 31);
      const R lam = __shfl_sync(0xffffffffu, lam_lane, gi & 31);
      const bool valid = gi < th.cnt;
      const long long b = valid ? lo : 0, e = valid ? hi : 0;
      double ss = 0.0;
#pragma unroll
      for (int j = 0; j < kEPL; ++j) {
        const long long i = b + (long long)j * L + sub;
        if (i < e) ss += term(ldv(xk + i), ldv(sj + i), ldv(y + i));
      }
      ss = sub_sum(ss, L);
      if (valid && sub == 0) p.s += (double)(lam * (R)sqrt_fast(ss));
      pos += 32 >> k;
    }
  }
  p = block_fold<kGroupThreads>(p);
  if (threadIdx.x == 0) partials[blockIdx.x] = p;
}

// ψ(y) of the CTA-per-group classes (see group_l2_big_kernel): xk | sj | y of a group arrive by bulk copies, ST groups
// in flight ahead of the one being summed
template <class R, int T, int LO, int EA, int EB, int ST>
__global__ void __launch_bounds__(T, 512 / T)
    group_value_big_kernel(const R* __restrict__ xk, const R* __restrict__ sj, const R* __restrict__ y, long long ngroups,
                           const long long* __restrict__ offs, const R* __restrict__ lambda_g, bool binf, double rad,
                           Partial* __restrict__ partials) {
  constexpr int PLS = bulk_plane<R>(EB * T);
  __shared__ int list[T];
  __shared__ int wcount[T / 32];
  __shared__ double red[T / 32];
  __shared__ __align__(8) uint64_t bar[ST];
  extern __shared__ __align__(128) unsigned char val_stage_raw[];
  const int t = threadIdx.x;
  StageRing<R, 3, PLS, ST> ring(bar, reinterpret_cast<R*>(val_stage_raw));  // xk | sj | y
  Partial p;
  p.s = 0.0;
  p.s2 = 0.0;
  p.bad = -1;
  for (long long g0 = (long long)blockIdx.x * T; g0 < ngroups; g0 += (long long)gridDim.x * T) {
    const int nbig = list_class_groups<T, LO, EB * T>(offs, g0, ngroups, list, wcount);
    ring.prime(list, nbig, g0, offs, xk, sj, y);
    for (int j = 0; j < nbig; ++j) {
      const long long g = g0 + list[j];
      const long long b = offs[g], e = offs[g + 1];
      const R* stage = ring.wait(j);
      const R* px = stage + bulk_skip(xk + b) + t;
      const R* ps = stage + PLS + bulk_skip(sj + b) + t;
      const R* py = stage + 2 * PLS + bulk_skip(y + b) + t;
      double ss = 0.0;
      const int ne = (e - b <= EA * T) ? EA : EB;
#pragma unroll
      for (int k = 0; k < EB; ++k) {
        const long long i = b + (long long)k * T + t;
        if (k < ne && i < e) {
          const R xi = px[k * T], si = ps[k * T], yi = py[k * T];
          R v;
          if (binf) {  // w = sj + y against the ball, v = w + xk  (shiftedGroupNormL2Binf.jl:34-39)
            const R w = si + yi;
            if ((double)w < -rad || (double)w > rad) p.bad = 1;
            v = w + xi;
          } else {
            v = (xi + si) + yi;  // ShiftedProximalOperators.jl:51-54
          }
          ss += (double)v * (double)v;
        }
      }
      ss = block_sum<T>(ss, red);
      if (t == 0) {
        long long ahead_b, ahead_e;
        if (ring.ahead(list, nbig, j, g0, offs, ahead_b, ahead_e)) ring.refill(xk, sj, y, ahead_b, ahead_e);
        p.s += (double)(lambda_g[g] * (R)sqrt(ss));  // λ_g ‖v_g‖  groupNormL2.jl:36
      }
    }
  }
  p = block_fold<T>(p);
  if (threadIdx.x == 0) partials[blockIdx.x] = p;
}

// ---- a single group spanning the whole vector (ShiftedGroupNormL2 built from NormL2, runtests.jl:244) ----
// One warp cannot stream a vector: the norm is a grid-wide reduction pass (3R), the scaling a second
// streaming pass (3R + 1W) on the elementwise kernel.
template <class R> struct SolSumSq {
  using Real = R;
  static constexpr int NIN = 3, UNROLL = 4;
  static constexpr bool OUT = false, ACC = true;
  const R* in[NIN];  // xk, sj, q
  R fill[NIN];
  R* y;
  __device__ __forceinline__ R apply(const R (&x)[NIN], long long, Partial& acc) const {
    const double s = (double)((x[2] + x[0]) + x[1]);
    acc.s2 += s * s;
    return R(0);
  }
};
// the same pass in the solver step: in[2] is ∇f and q = (-ν)∇f is rounded to R as it is read (same grid, same order)
template <class R> struct SolSumSqGrad : SolSumSq<R> {
  R mnu;
  __device__ __forceinline__ R apply(const R (&x)[3], long long, Partial& acc) const {
    const double s = (double)((mnu * x[2] + x[0]) + x[1]);
    acc.s2 += s * s;
    return R(0);
  }
};
template <class R> struct VSumSq {
  using Real = R;
  static constexpr int NIN = 3, UNROLL = 4;
  static constexpr bool OUT = false, ACC = true;
  const R* in[NIN];  // xk, sj, y
  R fill[NIN];
  R* y;
  bool binf;
  double rad;
  __device__ __forceinline__ R apply(const R (&x)[NIN], long long, Partial& acc) const {
    R v;
    if (binf) {
      const R w = x[1] + x[2];
      if ((double)w < -rad || (double)w > rad) acc.bad = 1;
      v = w + x[0];
    } else {
      v = (x[0] + x[1]) + x[2];
    }
    acc.s2 += (double)v * (double)v;
    return R(0);
  }
};
constexpr int64_t kSingleGroupMin = 1 << 15;  // below this one warp is quick enough

template <class Op, class R> static void set_in3(Op& op, const R* a, const R* b, const R* c) {
  op.in[0] = a; op.in[1] = b; op.in[2] = c;
  op.fill[0] = op.fill[1] = op.fill[2] = R(0);
  op.y = nullptr;
}

template <class R>
static int32_t prox_single_group(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q,
                                 const R* lambda_g, R sigma, double* psi_out) {
  R lam;
  SPX_CUDA(cudaMemcpyAsync(&lam, lambda_g, sizeof(R), cudaMemcpyDeviceToHost, ctx->stream));
  SolSumSq<R> ss;
  set_in3(ss, xk, sj, q);
  int nb = 0;
  int32_t st = ew_launch(ctx, ctx->stream, ss, n, 0, ctx->d_partials, &nb);
  if (st != SPX_OK) return st;
  st = finalize_partials(ctx, nb, 1, false);  // synchronises: lam has arrived as well
  if (st != SPX_OK) return st;
  const R snorm = (R)std::sqrt(ctx->h_result[0].s2);
  R alpha = R(1) - sigma * lam / snorm;  // shiftedGroupNormL2.jl:70-77
  alpha = (alpha != alpha) ? alpha : (alpha > R(0) ? alpha : R(0));
  if (psi_out) {
    SolScale<R, true> sc;
    set_in3(sc, xk, sj, q);
    sc.y = y; sc.alpha = alpha; sc.zero = snorm == R(0);
    st = ew_launch(ctx, ctx->stream, sc, n, 0, ctx->d_partials, &nb);
    if (st != SPX_OK) return st;
    st = finalize_partials(ctx, nb, 1, false);
    if (st != SPX_OK) return st;
    *psi_out = (double)(R)(double)(lam * (R)std::sqrt(ctx->h_result[0].s2));
    return SPX_OK;
  }
  SolScale<R, false> sc;
  set_in3(sc, xk, sj, q);
  sc.y = y; sc.alpha = alpha; sc.zero = snorm == R(0);
  return ew_launch(ctx, ctx->stream, sc, n, 0, ctx->d_partials, &nb);
}

// Grid of `want` CTAs, clamped to [1, cap].  A persistent (grid-stride) kernel is also held to the CTAs the device keeps
// resident at once; a short-lived one (one CTA per chunk of work, cap kGridMax) is not.  Dynamic shared memory above
// the default limit has to be allowed before the occupancy query and the launch.
constexpr long long kGridMax = 1 << 20;
static int32_t grid_for(spx_ctx* ctx, const void* kernel, int threads, size_t smem, long long want, long long cap,
                        bool persistent, int* grid) {
  if (smem > 0) SPX_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (persistent) {
    int per_sm = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem) != cudaSuccess || per_sm < 1)
      per_sm = 1;
    cap = std::min(cap, (long long)ctx->sm_count * per_sm);
  }
  *grid = (int)std::max(1LL, std::min(want, cap));
  return SPX_OK;
}
// CTAs of a warp kernel (256 threads, one warp per task of kTask groups) that give every warp one task
static long long warp_kernel_ctas(int64_t ngroups) {
  const long long ntasks = (ngroups + kTask - 1) / kTask;
  return (ntasks + (kGroupThreads / 32) - 1) / (kGroupThreads / 32);
}
// grid of a persistent warp kernel: one task per warp, at most the resident CTAs and kMaxPartials
static int32_t group_grid(spx_ctx* ctx, int64_t ngroups, const void* kernel, int* grid) {
  return grid_for(ctx, kernel, kGroupThreads, 0, warp_kernel_ctas(ngroups), kMaxPartials, true, grid);
}

// what spx_group_validate_offsets recorded for this layout, or nullptr
static const spx_ctx::GroupCensus* find_census(const spx_ctx* ctx, const void* offs, int64_t ngroups, int64_t n) {
  for (const auto& c : ctx->census)
    if (c.offs == offs && c.ngroups == (long long)ngroups && c.n == (long long)n) return &c;
  return nullptr;
}
// classes to launch for this layout: what the census recorded, both when the layout is unknown
static unsigned census_classes(const spx_ctx* ctx, const void* offs, int64_t ngroups, int64_t n) {
  const spx_ctx::GroupCensus* c = find_census(ctx, offs, ngroups, n);
  return c ? c->classes & 3u : 3u;
}

// The context's side streams 0 and 1 and three events, created on first use: fork_side_streams makes both streams wait
// for the work enqueued so far on ctx->stream, join_side_streams makes ctx->stream wait for both.
static int32_t fork_side_streams(spx_ctx* ctx) {
  for (int i = 0; i < 2; ++i)
    if (!ctx->pipe_streams[i]) SPX_CUDA(cudaStreamCreateWithFlags(&ctx->pipe_streams[i], cudaStreamNonBlocking));
  for (cudaEvent_t& ev : ctx->pipe_events)
    if (!ev) SPX_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  SPX_CUDA(cudaEventRecord(ctx->pipe_events[0], ctx->stream));
  for (int i = 0; i < 2; ++i) SPX_CUDA(cudaStreamWaitEvent(ctx->pipe_streams[i], ctx->pipe_events[0], 0));
  return SPX_OK;
}
static int32_t join_side_streams(spx_ctx* ctx) {
  for (int i = 0; i < 2; ++i) {
    SPX_CUDA(cudaEventRecord(ctx->pipe_events[1 + i], ctx->pipe_streams[i]));
    SPX_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->pipe_events[1 + i], 0));
  }
  return SPX_OK;
}

#ifndef SPX_L2_MID_STAGES
#define SPX_L2_MID_STAGES 2
#endif
// grid of a persistent CTA-per-group kernel: one CTA per chunk of `threads` groups, at most the resident CTAs
static int32_t big_grid(spx_ctx* ctx, int64_t ngroups, const void* kernel, int threads, size_t stage_bytes, int* grid) {
  return grid_for(ctx, kernel, threads, stage_bytes, (ngroups + threads - 1) / threads, kMaxPartials / 4, true, grid);
}

template <class R>
int32_t value_group_binf(spx_ctx* ctx, int64_t n, const R* xk, const R* sj, const R* y, bool binf, double delta,
                         int64_t ngroups, const int64_t* offs, const R* lambda_g, double* out) {
  SPX_REQUIRE(ctx && out, "null argument");
  SPX_REQUIRE(n >= 0 && ngroups >= 0, "negative size");
  SPX_REQUIRE(ngroups == 0 || (offs && lambda_g && xk && sj && y), "null device vector");
  DeviceGuard g(ctx->device);
  if (ngroups == 0) {
    *out = 0.0;
    return SPX_OK;
  }
  if (ngroups == 1 && n >= kSingleGroupMin) {  // one group spanning the vector: grid-wide reduction
    R lam;
    SPX_CUDA(cudaMemcpyAsync(&lam, lambda_g, sizeof(R), cudaMemcpyDeviceToHost, ctx->stream));
    VSumSq<R> op;
    set_in3(op, xk, sj, y);
    op.binf = binf;
    op.rad = 1.1 * (double)(R)delta;
    int nb = 0;
    int32_t st1 = ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, &nb);
    if (st1 != SPX_OK) return st1;
    st1 = finalize_partials(ctx, nb, 1, false);
    if (st1 != SPX_OK) return st1;
    *out = ctx->h_result[0].bad > 0 ? std::numeric_limits<double>::infinity()
                                    : (double)(R)(double)(lam * (R)std::sqrt(ctx->h_result[0].s2));
    return SPX_OK;
  }
  const double rad = 1.1 * (double)(R)delta;
  int grid0 = 0, grid1 = 0, grid2 = 0, grid3 = 0;
  int32_t st = group_grid(ctx, ngroups, (const void*)group_value_kernel<R, 0>, &grid0);
  if (st == SPX_OK) st = group_grid(ctx, ngroups, (const void*)group_value_kernel<R, 1>, &grid1);
  // the classes (256, 1024] and (1024, 4096]: CTA per group, operands by bulk copies (as in launch_group_l2)
  constexpr int kMidT = 128;
  auto big_val = group_value_big_kernel<R, kGroupThreads, (int)kBigMin, kBigE / 2, kBigE, 1>;
  auto mid_val = group_value_big_kernel<R, kMidT, (int)kMidMin, 4, 8, SPX_L2_MID_STAGES>;
  const size_t big_bytes = 3 * (size_t)bulk_plane<R>((int)kBigMax) * sizeof(R);
  const size_t mid_bytes = SPX_L2_MID_STAGES * 3 * (size_t)bulk_plane<R>((int)kBigMin) * sizeof(R);
  const unsigned classes = census_classes(ctx, offs, ngroups, n);
  if (st == SPX_OK && (classes & 2u)) st = big_grid(ctx, ngroups, (const void*)big_val, kGroupThreads, big_bytes, &grid2);
  if (st == SPX_OK && (classes & 1u)) st = big_grid(ctx, ngroups, (const void*)mid_val, kMidT, mid_bytes, &grid3);
  if (st != SPX_OK) return st;
  group_value_kernel<R, 0><<<grid0, kGroupThreads, 0, ctx->stream>>>(xk, sj, y, ngroups, (const long long*)offs, lambda_g,
                                                                    binf, rad, classes, ctx->d_partials);
  group_value_kernel<R, 1><<<grid1, kGroupThreads, 0, ctx->stream>>>(xk, sj, y, ngroups, (const long long*)offs, lambda_g,
                                                                    binf, rad, classes, ctx->d_partials + grid0);
  if (grid2 > 0)
    big_val<<<grid2, kGroupThreads, big_bytes, ctx->stream>>>(xk, sj, y, ngroups, (const long long*)offs, lambda_g, binf,
                                                             rad, ctx->d_partials + grid0 + grid1);
  if (grid3 > 0)
    mid_val<<<grid3, kMidT, mid_bytes, ctx->stream>>>(xk, sj, y, ngroups, (const long long*)offs, lambda_g, binf, rad,
                                                     ctx->d_partials + grid0 + grid1 + grid2);
  ctx->launches += 2 + (grid2 > 0) + (grid3 > 0);
  SPX_CUDA(cudaGetLastError());
  st = finalize_partials(ctx, grid0 + grid1 + grid2 + grid3, 1, false);
  if (st != SPX_OK) return st;
  // the reference accumulates sum_c in R; one rounding to R here
  *out = ctx->h_result[0].bad > 0 ? std::numeric_limits<double>::infinity() : (double)(R)ctx->h_result[0].s;
  return SPX_OK;
}
template int32_t value_group_binf<double>(spx_ctx*, int64_t, const double*, const double*, const double*, bool, double,
                                          int64_t, const int64_t*, const double*, double*);
template int32_t value_group_binf<float>(spx_ctx*, int64_t, const float*, const float*, const float*, bool, double,
                                         int64_t, const int64_t*, const float*, double*);

template <class R, bool SHIFTED>
static int32_t launch_group_l2(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q, int64_t ngroups,
                               const int64_t* offs, const R* lambda_g, R sigma, double* psi_out) {
  const unsigned classes = census_classes(ctx, offs, ngroups, n);
  // The CTA-per-group classes stage q | xk | sj in shared memory with bulk copies: (1024, 4096] with 256 threads and one
  // buffer (the copy of the next group runs under the stores of the current one; two CTAs per SM overlap the rest),
  // (256, 1024] with 128 threads and a ring of two buffers (four CTAs per SM; a ring of four with two CTAs measured 3 % slower).
  constexpr int kMidT = 128, kMidStages = SPX_L2_MID_STAGES, NP = SHIFTED ? 3 : 1;
  const size_t big_bytes = NP * (size_t)bulk_plane<R>((int)kBigMax) * sizeof(R);
  const size_t mid_bytes = kMidStages * NP * (size_t)bulk_plane<R>((int)kBigMin) * sizeof(R);
  auto big_psi = group_l2_big_kernel<R, true, SHIFTED, kGroupThreads, (int)kBigMin, kBigE / 2, kBigE, 1>;
  auto big_run = group_l2_big_kernel<R, false, SHIFTED, kGroupThreads, (int)kBigMin, kBigE / 2, kBigE, 1>;
  auto mid_psi = group_l2_big_kernel<R, true, SHIFTED, kMidT, (int)kMidMin, 4, 8, kMidStages>;
  auto mid_run = group_l2_big_kernel<R, false, SHIFTED, kMidT, (int)kMidMin, 4, 8, kMidStages>;
  if (psi_out) {
    int grid0 = 0, grid1 = 0, grid2 = 0, grid3 = 0;
    int32_t st = group_grid(ctx, ngroups, (const void*)group_l2_kernel<R, true, 0, SHIFTED>, &grid0);
    if (st == SPX_OK) st = group_grid(ctx, ngroups, (const void*)group_l2_kernel<R, true, 1, SHIFTED>, &grid1);
    if (st == SPX_OK && (classes & 2u)) st = big_grid(ctx, ngroups, (const void*)big_psi, kGroupThreads, big_bytes, &grid2);
    if (st == SPX_OK && (classes & 1u)) st = big_grid(ctx, ngroups, (const void*)mid_psi, kMidT, mid_bytes, &grid3);
    if (st != SPX_OK) return st;
    group_l2_kernel<R, true, 0, SHIFTED><<<grid0, kGroupThreads, 0, ctx->stream>>>(
        y, xk, sj, q, ngroups, (const long long*)offs, lambda_g, sigma, classes, ctx->d_partials, nullptr, R(0), nullptr);
    group_l2_kernel<R, true, 1, SHIFTED><<<grid1, kGroupThreads, 0, ctx->stream>>>(
        y, xk, sj, q, ngroups, (const long long*)offs, lambda_g, sigma, classes, ctx->d_partials + grid0, nullptr, R(0),
        nullptr);
    if (grid2 > 0)
      big_psi<<<grid2, kGroupThreads, big_bytes, ctx->stream>>>(y, xk, sj, q, ngroups, (const long long*)offs, lambda_g,
                                                               sigma, ctx->d_partials + grid0 + grid1, nullptr, R(0), nullptr);
    if (grid3 > 0)
      mid_psi<<<grid3, kMidT, mid_bytes, ctx->stream>>>(y, xk, sj, q, ngroups, (const long long*)offs, lambda_g, sigma,
                                                       ctx->d_partials + grid0 + grid1 + grid2, nullptr, R(0), nullptr);
    ctx->launches += 2 + (grid2 > 0) + (grid3 > 0);
    SPX_CUDA(cudaGetLastError());
    st = finalize_partials(ctx, grid0 + grid1 + grid2 + grid3, 1, false);
    if (st != SPX_OK) return st;
    *psi_out = (double)(R)ctx->h_result[0].s;
    return SPX_OK;
  }
  // The size classes are independent: they run CONCURRENTLY on the context's side streams (fork / join by events on
  // the caller's stream), with one short-lived CTA per chunk of work instead of a persistent grid, so the block
  // scheduler interleaves the kernels as resources free up (the short-group class waits on its per-group arithmetic).
  int grid0 = 0, grid2 = 0, grid3 = 0;
  int32_t st = grid_for(ctx, (const void*)group_l2_kernel<R, false, 0, SHIFTED>, kGroupThreads, 0,
                        warp_kernel_ctas(ngroups), kGridMax, false, &grid0);
  // A class the layout is known not to hold (census of spx_group_validate_offsets) is not launched: its CTAs would
  // only scan the offsets, but their shared-memory carve-out keeps the warp kernel off the SMs they pass through
  // (uniform groups of 64: 2.21 ms with the two empty launches, 1.44 ms without).
  if (st == SPX_OK && (classes & 2u))
    st = grid_for(ctx, (const void*)big_run, kGroupThreads, big_bytes, (ngroups + kGroupThreads - 1) / kGroupThreads,
                  kGridMax, false, &grid2);
  if (st == SPX_OK && (classes & 1u))
    st = grid_for(ctx, (const void*)mid_run, kMidT, mid_bytes, (ngroups + kMidT - 1) / kMidT, kGridMax, false, &grid3);
  if (st == SPX_OK) st = fork_side_streams(ctx);
  if (st != SPX_OK) return st;
  if (grid2 > 0) {
    big_run<<<grid2, kGroupThreads, big_bytes, ctx->stream>>>(y, xk, sj, q, ngroups, (const long long*)offs, lambda_g,
                                                             sigma, ctx->d_partials, nullptr, R(0), nullptr);
    ctx->launches++;
  }
  if (grid3 > 0) {
    mid_run<<<grid3, kMidT, mid_bytes, ctx->pipe_streams[0]>>>(y, xk, sj, q, ngroups, (const long long*)offs, lambda_g,
                                                              sigma, ctx->d_partials, nullptr, R(0), nullptr);
    ctx->launches++;
  }
  // groups above 4096 elements (and those of a class not launched): the warp path, whose CTAs exit at once when there
  // are none -- on the side stream, under the short-group kernel
  group_l2_kernel<R, false, 1, SHIFTED><<<grid0, kGroupThreads, 0, ctx->pipe_streams[1]>>>(
      y, xk, sj, q, ngroups, (const long long*)offs, lambda_g, sigma, classes, ctx->d_partials, nullptr, R(0), nullptr);
  group_l2_kernel<R, false, 0, SHIFTED><<<grid0, kGroupThreads, 0, classes == 0u ? ctx->stream : ctx->pipe_streams[1]>>>(
      y, xk, sj, q, ngroups, (const long long*)offs, lambda_g, sigma, classes, ctx->d_partials, nullptr, R(0), nullptr);
  ctx->launches += 2;
  SPX_CUDA(cudaGetLastError());
  return join_side_streams(ctx);
}

// the operands of the step form of the uniform kernels (spx_step_groupl2binf); nblocks returns the CTAs of both
// launches, whose two partial slots each lie at d_partials[k * nblocks ...]
template <class R> struct UniformStep {
  R* xsy;
  R mnu;
  double rad;
  unsigned char* declined;
  int nblocks;
};

template <class R, int L, bool STEP>
static int32_t launch_uniform_binf_L(spx_ctx* ctx, R* y, const R* xk, const R* sj, const R* q, int64_t ngroups,
                                     const R* lambda_g, R sigma, R delta, UDiv<R> by_sigma, const unsigned* uniform_flag,
                                     unsigned* wl_count, unsigned* wl_rounds, UniformStep<R>* step) {
  const long long nrounds = (ngroups + (32 / L) - 1) / (32 / L);
  const long long want = (nrounds + (kGroupThreads / 32) - 1) / (kGroupThreads / 32);
  const size_t smem = (size_t)(kGroupThreads / 32) * UTile<R, L>::kWarpBytes;
  auto fast = group_l2binf_uniform_kernel<R, L, true, STEP>;
  auto list = group_l2binf_uniform_kernel<R, L, false, STEP>;
  int grid_fast = 0, grid_list = 0;
  int32_t st = grid_for(ctx, (const void*)fast, kGroupThreads, smem, want, kGridMax, true, &grid_fast);
  if (st == SPX_OK) st = grid_for(ctx, (const void*)list, kGroupThreads, smem, want, kGridMax, true, &grid_list);
  if (st != SPX_OK) return st;
  UniformStep<R> a{nullptr, R(0), 0.0, nullptr, 0};
  Partial *p0 = nullptr, *p1 = nullptr;
  if constexpr (STEP) {
    step->nblocks = grid_fast + grid_list;
    a = *step;
    p0 = ctx->d_partials;
    p1 = ctx->d_partials + step->nblocks;
  }
  fast<<<grid_fast, kGroupThreads, smem, ctx->stream>>>(y, xk, sj, q, ngroups, lambda_g, sigma, delta, by_sigma,
                                                        uniform_flag, wl_count, wl_rounds, a.xsy, a.mnu, a.rad,
                                                        a.declined, p0, p1);
  list<<<grid_list, kGroupThreads, smem, ctx->stream>>>(y, xk, sj, q, ngroups, lambda_g, sigma, delta, by_sigma,
                                                        uniform_flag, wl_count, wl_rounds, a.xsy, a.mnu, a.rad,
                                                        a.declined, STEP ? p0 + grid_fast : nullptr,
                                                        STEP ? p1 + grid_fast : nullptr);
  return SPX_OK;
}
template <class R, bool STEP = false>
static int32_t launch_uniform_binf(spx_ctx* ctx, int L, R* y, const R* xk, const R* sj, const R* q, int64_t ngroups,
                                   const R* lambda_g, R sigma, R delta, UDiv<R> by_sigma, const unsigned* uniform_flag,
                                   unsigned* wl_count, unsigned* wl_rounds, UniformStep<R>* step = nullptr) {
  switch (L) {
#define SPX_UL(LL)                                                                                                   \
  case LL:                                                                                                           \
    return launch_uniform_binf_L<R, LL, STEP>(ctx, y, xk, sj, q, ngroups, lambda_g, sigma, delta, by_sigma,         \
                                              uniform_flag, wl_count, wl_rounds, step);
    SPX_UL(2) SPX_UL(4) SPX_UL(8) SPX_UL(16) SPX_UL(32)
#undef SPX_UL
    default: return SPX_OK;
  }
}

// The uniform kernels' conditions that the host can check (whether offs is {0, m, 2m, ...} is checked on the device):
// n == ngroups m with m = 8 L, 16-byte aligned vectors, and σ, Δ far enough inside the normal range for the fast
// searches' branch-free quotients (sol/σ).
static bool binf_sigma_ok(double sigma, double delta) {
  return std::isfinite(sigma) && std::fabs(sigma) > 1e-30 && std::fabs(sigma) < 1e30 && std::isfinite(delta) &&
         std::fabs(delta) < 1e30;
}
static bool uniform_binf_candidate(int64_t n, int64_t m, bool aligned, double sigma, double delta) {
  return binf_sigma_ok(sigma, delta) && aligned && (m == 16 || m == 32 || m == 64 || m == 128 || m == 256) &&
         n < (int64_t(1) << 39);
}

// ctx->d_scratch during a GroupNormL2Binf prox!: a head that every call clears, the work list of the uniform kernels at
// 4 KiB, then `done` (one byte per group) on the next 256-byte boundary behind the list
struct BinfScratch {
  struct alignas(32) Head {
    unsigned long long counter;  // task hand-out of the long groups (group_l2binf_kernel<R, 1>)
    unsigned long_flag;          // some task holds a group of more than 256 elements
    unsigned uniform_flag;       // offs is {0, m, 2m, ...}: the uniform kernels own the call
    unsigned wl_count;           // rounds in wl_rounds
  } head;
  unsigned char unused[4096 - sizeof(Head)];
  unsigned wl_rounds[1];  // one entry per round of the uniform layout
  static size_t done_offset(int64_t nrounds) {
    return offsetof(BinfScratch, wl_rounds) + (((size_t)nrounds * sizeof(unsigned) + 255) & ~(size_t)255);
  }
};
static_assert(sizeof(BinfScratch::Head) == 32 && offsetof(BinfScratch, wl_rounds) == 4096, "Binf scratch layout");

template <class R>
static int32_t prox_group(spx_ctx* ctx, bool binf, int64_t n, R* y, const R* xk, const R* sj, const R* q,
                          int64_t ngroups, const int64_t* offs, const R* lambda_g, double sigma, double delta,
                          double* psi_out) {
  SPX_REQUIRE(ctx != nullptr, "null context");
  SPX_REQUIRE(n >= 0 && ngroups >= 0, "negative size");
  SPX_REQUIRE(ngroups == 0 || (y && q && offs && lambda_g), "null device vector");
  SPX_REQUIRE((xk == nullptr) == (sj == nullptr), "xk and sj must both be given or both be NULL");
  SPX_REQUIRE(!(binf && ngroups > 0 && xk == nullptr), "the Binf form needs its shifts");
  DeviceGuard g(ctx->device);
  if (ngroups == 1 && !binf && xk != nullptr && n >= kSingleGroupMin) return prox_single_group<R>(ctx, n, y, xk, sj, q, lambda_g, (R)sigma, psi_out);
  if (ngroups > 0) {
    if (!binf) {
      return xk ? launch_group_l2<R, true>(ctx, n, y, xk, sj, q, ngroups, offs, lambda_g, (R)sigma, psi_out)
                : launch_group_l2<R, false>(ctx, n, y, xk, sj, q, ngroups, offs, lambda_g, (R)sigma, psi_out);
    }
    UDiv<R> by_sigma;
    by_sigma.set((R)sigma);
    int grid0 = 0, grid1 = 0;
    int32_t st = group_grid(ctx, ngroups, (const void*)group_l2binf_kernel<R, 0>, &grid0);
    if (st == SPX_OK) st = group_grid(ctx, ngroups, (const void*)group_l2binf_kernel<R, 1>, &grid1);
    if (st != SPX_OK) return st;
    // uniform layout candidate: n == ngroups m, m = 8 L, 16-byte aligned vectors.  Whether offs really is
    // {0, m, 2m, ...} is checked on the device; the flag gates the uniform kernels and the generic ones.
    const int64_t m = ngroups > 0 && n % ngroups == 0 ? n / ngroups : 0;
    const bool aligned = (((uintptr_t)y | (uintptr_t)xk | (uintptr_t)sj | (uintptr_t)q) & 15u) == 0;
    // the fast searches take sol/σ through the branch-free quotient: σ far inside the normal range only
    const bool sigma_ok = binf_sigma_ok(sigma, delta);
    const bool uni = uniform_binf_candidate(n, m, aligned, sigma, delta);
    const size_t done_off = BinfScratch::done_offset(uni ? (n + kRoundElems - 1) / kRoundElems : 0);
    st = ensure_scratch(ctx, done_off + (size_t)ngroups + 256);
    if (st != SPX_OK) return st;
    BinfScratch* const scratch = (BinfScratch*)ctx->d_scratch;
    unsigned* const uniform_flag = &scratch->head.uniform_flag;
    SPX_CUDA(cudaMemsetAsync(&scratch->head, 0, sizeof(BinfScratch::Head), ctx->stream));
    if (uni) {
      SPX_CUDA(cudaMemsetAsync(uniform_flag, 1, sizeof(unsigned), ctx->stream));
      const int cgrid = (int)std::min<int64_t>((ngroups + 256) / 256, (int64_t)ctx->sm_count * 8);
      group_uniform_check_kernel<<<cgrid, 256, 0, ctx->stream>>>((const long long*)offs, ngroups, m, uniform_flag);
      st = launch_uniform_binf<R>(ctx, (int)(m / kEPL), y, xk, sj, q, ngroups, lambda_g, (R)sigma, (R)delta, by_sigma,
                                  uniform_flag, &scratch->head.wl_count, scratch->wl_rounds);
      if (st != SPX_OK) return st;
      ctx->launches += 3;
    }
    // Fast kernels first, each marking the groups it has written in `done`: groups of <= 256 elements on the planner's
    // warp rounds, (1024, 4096] with 256 threads per group, (256, 1024] with 128.  The bracketing search (the two warp
    // kernels) then takes whatever is left.  prox!(y, ψ, y, σ) (y IS an input vector) takes the same kernels as the
    // out-of-place call, so both give the same bits: every kernel reads a group's inputs before it writes that group's
    // y, a group is written by exactly one kernel, and a group a fast kernel declines is left untouched.  Not when y
    // overlaps an input partially (a group's y would land on another group's inputs) or σ, Δ are outside the range of
    // the branch-free quotient.
    unsigned char* done = nullptr;
    auto overlaps = [&](const R* p) { return p != y && spans_overlap(y, p, (size_t)n * sizeof(R)); };
    if (sigma_ok && !(overlaps(xk) || overlaps(sj) || overlaps(q))) {
      done = (unsigned char*)ctx->d_scratch + done_off;
      SPX_CUDA(cudaMemsetAsync(done, 0, (size_t)ngroups, ctx->stream));
      // a class the layout is known not to hold is not launched (whatever is not marked done goes to the bracketing
      // search anyway, so the census is only a hint here as well)
      const unsigned classes = census_classes(ctx, offs, ngroups, n);
      // With CTA-per-group classes present the fast kernels run CONCURRENTLY (short groups and the 128-thread classes on
      // the context's side streams, as in launch_group_l2), each with one short-lived CTA per chunk of groups instead of
      // a persistent grid: the block scheduler then mixes CTAs of the kernels on an SM, and the barrier-separated phases
      // of one kernel leave their idle issue slots to the others.
      const bool fork = classes != 0u;
      if (fork) {
        st = fork_side_streams(ctx);
        if (st != SPX_OK) return st;
      }
      auto launch_class = [&](auto kern, int threads, size_t stage_bytes, cudaStream_t stream) -> int32_t {
        int grid = 0;
        const int32_t s2 = grid_for(ctx, (const void*)kern, threads, stage_bytes, (ngroups + threads - 1) / threads,
                                    kGridMax, false, &grid);
        if (s2 != SPX_OK) return s2;
        kern<<<grid, threads, stage_bytes, stream>>>(y, xk, sj, q, ngroups, (const long long*)offs, lambda_g, (R)sigma,
                                                     (R)delta, by_sigma, uni ? uniform_flag : nullptr, done);
        ctx->launches++;
        return SPX_OK;
      };
      // (1024, 4096]: 256 threads x 8 or 16 elements, two CTAs per SM in 128 registers (measured at 2^28 Float64,
      // ragged layout: 2.8 ms; split into 512 x 8 and 256 x 8 at 64 registers and 1024 threads per SM: 3.4 ms;
      // three CTAs per SM in 80 registers with sj read from global memory instead of staged: 3.3 ms -- more
      // resident CTAs do not help this class).
      // (256, 1024]: two shapes of 128 threads, 8 and 4 elements, 64 registers (0.77 ms; one shape of 4 or 8
      // elements at 128 registers: 0.94 ms).
      if (classes & 2u) {
        st = launch_class(group_l2binf_big_kernel<R, kBinfBigThreads, 1024, 8, 16, 512>, kBinfBigThreads,
                          3 * (size_t)bulk_plane<R>(16 * kBinfBigThreads) * sizeof(R), ctx->stream);
        if (st != SPX_OK) return st;
      }
      if (classes & 1u) {
        st = launch_class(group_l2binf_big_kernel<R, kBinfMidThreads, 512, 8, 8, 1024>, kBinfMidThreads,
                          3 * (size_t)bulk_plane<R>(8 * kBinfMidThreads) * sizeof(R), ctx->pipe_streams[0]);
        if (st != SPX_OK) return st;
        st = launch_class(group_l2binf_big_kernel<R, kBinfMidThreads, 256, 4, 4, 1024>, kBinfMidThreads,
                          3 * (size_t)bulk_plane<R>(4 * kBinfMidThreads) * sizeof(R), ctx->pipe_streams[0]);
        if (st != SPX_OK) return st;
      }
      // the short groups last: the class (1024, 4096] is the long pole and should get the SMs first.  Alone (no class
      // present) they take a persistent grid on ctx->stream.
      int grids = 0;
      st = grid_for(ctx, (const void*)group_l2binf_small_fast_kernel<R>, kGroupThreads, 0, warp_kernel_ctas(ngroups),
                    fork ? kGridMax : kMaxPartials, !fork, &grids);
      if (st != SPX_OK) return st;
      group_l2binf_small_fast_kernel<R><<<grids, kGroupThreads, 0, fork ? ctx->pipe_streams[1] : ctx->stream>>>(
          y, xk, sj, q, ngroups, (const long long*)offs, lambda_g, (R)sigma, (R)delta, by_sigma,
          uni ? uniform_flag : nullptr, done);
      ctx->launches++;
      if (fork) {
        st = join_side_streams(ctx);
        if (st != SPX_OK) return st;
      }
    }
    group_l2binf_kernel<R, 0><<<grid0, kGroupThreads, 0, ctx->stream>>>(
        y, xk, sj, q, ngroups, (const long long*)offs, lambda_g, (R)sigma, (R)delta, by_sigma, nullptr,
        &scratch->head.long_flag, uni ? uniform_flag : nullptr, done);
    group_l2binf_kernel<R, 1><<<grid1, kGroupThreads, 0, ctx->stream>>>(
        y, xk, sj, q, ngroups, (const long long*)offs, lambda_g, (R)sigma, (R)delta, by_sigma, &scratch->head.counter,
        &scratch->head.long_flag, uni ? uniform_flag : nullptr, done);
    ctx->launches += 2;
    SPX_CUDA(cudaGetLastError());
  }
  if (psi_out) {
    if (!binf) {
      *psi_out = 0.0;
      return SPX_OK;
    }
    // the trust-region value needs sj + y and xk separately: one more streaming pass
    return value_group_binf<R>(ctx, n, xk, sj, y, true, delta, ngroups, offs, lambda_g, psi_out);
  }
  return SPX_OK;
}

// ---- the solver step of ShiftedGroupNormL2 (SURVEY.md 8f rank 1; spx_step.cu for the separable types) ---------------
//     q = (-ν) ∇f;  prox!(s, ψ, q, ν);  xsy = (xk + sj) + s;  ψ(s);  Σ s²;  Σ ∇f·s
// Every layout runs it in the passes of the prox! kernels of its group sizes, with ∇f in place of q on the load (q =
// (-ν)∇f rounded to R, as the caller's broadcast would) and a store loop that also writes xsy and folds the two sums next
// to the ψ term: s is bit for bit what prox! writes.  Groups of <= 256 elements take the packed warp rounds of
// group_l2_step_kernel (on a validated layout without longer groups, the C4 shape, alone: one launch and the fold), the
// CTA-per-group classes the step forms of group_l2_big_kernel, longer groups the step form of the warp path
// (group_l2_kernel<…, PART 1>), and a single group spanning the vector the two grid-wide passes of prox_single_group.
// group_l2_step_kernel: two CTAs per SM (125 registers in Float64: sol, ∇f and xk + sj of 8 elements per lane); three
// spill and measure the same (2.60 vs 2.54 ms at 2^28 Float64).  long_runs: the long-group kernels run in the same call,
// so a group of more than 256 elements is theirs; without them such a group (a stale census) raises the flag.
#ifndef SPX_GSTEP_MINB
#define SPX_GSTEP_MINB 2
#endif
template <class R>
__global__ void __launch_bounds__(kGroupThreads, SPX_GSTEP_MINB)
    group_l2_step_kernel(R* s, R* xsy, const R* xk, const R* sj, const R* grad, long long ngroups,
                         const long long* __restrict__ offs, const R* __restrict__ lambda_g, R sigma, R mnu,
                         Partial* __restrict__ partials, Partial* __restrict__ part1, bool long_runs) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * kGroupThreads + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * kGroupThreads) >> 5;
  const long long ntasks = (ngroups + kTask - 1) / kTask;
  double psi = 0.0, ss2 = 0.0, dot = 0.0;
  long long bad = -1;
  for (long long task = warp; task < ntasks; task += nwarps) {
    const long long g0 = task * kTask;
    const TaskHead th = load_task(offs, g0, ngroups, lane);
    const R lam_lane = lane < th.cnt ? lambda_g[g0 + lane] : R(0);
    int pos = 0;
    while (pos < th.cnt) {
      const int k = plan_round(th.le, pos);
      if (k < 0) {  // a group of more than 256 elements: the long-group kernels' (flagged when they do not run)
        if (!long_runs) bad = 1;
        pos += 1;
        continue;
      }
      const int L = 1 << k, sub = lane & (L - 1), gi = pos + (lane >> k);
      const long long lo = __shfl_sync(0xffffffffu, th.lo, gi & 31), hi = __shfl_sync(0xffffffffu, th.hi, gi & 31);
      const R lam = __shfl_sync(0xffffffffu, lam_lane, gi & 31);
      const bool valid = gi < th.cnt;
      const long long b = valid ? lo : 0, e = valid ? hi : 0;
      R sol[kEPL], g[kEPL], xs[kEPL];
#pragma unroll
      for (int j = 0; j < kEPL; ++j) {
        const long long i = b + (long long)j * L + sub;
        sol[j] = R(0);
        g[j] = R(0);
        xs[j] = R(0);
        if (i < e) {
          const R xi = ldv(xk + i), si = ldv(sj + i), gj = ldv(grad + i);
          const R qi = mnu * gj;     // q = -ν ∇f
          sol[j] = (qi + xi) + si;   // shiftedGroupNormL2.jl:65
          xs[j] = xi + si;
          g[j] = gj;
        }
      }
      double ss = 0.0;
#pragma unroll
      for (int j = 0; j < kEPL; ++j) ss += (double)sol[j] * (double)sol[j];
      ss = sub_sum(ss, L);
      const R snorm = (R)sqrt_fast(ss);
      const R alpha = jl_max(R(1) - sigma * lam / snorm, R(0));
      double vv = 0.0;
#pragma unroll
      for (int j = 0; j < kEPL; ++j) {
        const long long i = b + (long long)j * L + sub;
        if (i < e) {
          const R o = (snorm == R(0) ? R(0) : alpha * sol[j]) - xs[j];  // :70-77
          stv(s + i, o);
          const R v = xs[j] + o;  // ψ's own argument (ShiftedProximalOperators.jl:52)
          if (xsy != nullptr) stv(xsy + i, v);
          vv += (double)v * (double)v;
          ss2 = __fma_rn((double)o, (double)o, ss2);
          dot = __fma_rn((double)g[j], (double)o, dot);
        }
      }
      vv = sub_sum(vv, L);
      if (valid && sub == 0) psi += (double)(lam * (R)sqrt_fast(vv));  // λ_g ‖v_g‖  groupNormL2.jl:36
      pos += 32 >> k;
    }
  }
  Partial p;
  p.s = psi;
  p.s2 = ss2;
  p.bad = bad;
  p = block_fold<kGroupThreads>(p);
  Partial p2;
  p2.s = dot;
  p2.s2 = 0.0;
  p2.bad = -1;
  p2 = block_fold<kGroupThreads>(p2);
  if (threadIdx.x == 0) {
    partials[blockIdx.x] = p;
    part1[blockIdx.x] = p2;
  }
}

// The step kernels of every group above 256 elements -- the CTA-per-group classes in `classes` and the warp kernel for
// the others -- and, with `short_groups`, group_l2_step_kernel for the rest, on persistent grids capped so that their
// CTAs together stay within kMaxPartials.  Kernel k writes slot 0 at d_partials + base_k and slot 1 at d_partials +
// total + base_k, so finalize_partials(ctx, total, 2) folds them in a fixed order: two identical calls give identical
// sums.  With a class present the kernels run on the context's side streams, as the plain prox! does (ragged 1..4096 on
// a B200: 2.72 against 2.97 ms at 2^28 Float64 with every kernel on ctx->stream, 3.20 against 3.37 ms at 2^29 Float32).
template <class R>
static int32_t launch_step_groupl2(spx_ctx* ctx, bool short_groups, unsigned classes, R* s, R* xsy, const R* xk,
                                   const R* sj, const R* grad, int64_t ngroups, const int64_t* offs, const R* lambda_g,
                                   R nu, int* total) {
  constexpr int kMidT = 128, kMidStages = SPX_L2_MID_STAGES, kCap = kMaxPartials / 4;
  const size_t big_bytes = 3 * (size_t)bulk_plane<R>((int)kBigMax) * sizeof(R);
  const size_t mid_bytes = kMidStages * 3 * (size_t)bulk_plane<R>((int)kBigMin) * sizeof(R);
  auto big = group_l2_big_kernel<R, true, true, kGroupThreads, (int)kBigMin, kBigE / 2, kBigE, 1, true>;
  auto mid = group_l2_big_kernel<R, true, true, kMidT, (int)kMidMin, 4, 8, kMidStages, true>;
  auto lng = group_l2_kernel<R, true, 1, true, true>;
  int gs = 0, gl = 0, gb = 0, gm = 0;
  int32_t st = SPX_OK;
  if (short_groups)
    st = grid_for(ctx, (const void*)group_l2_step_kernel<R>, kGroupThreads, 0, warp_kernel_ctas(ngroups), kCap, true, &gs);
  if (st == SPX_OK) st = grid_for(ctx, (const void*)lng, kGroupThreads, 0, warp_kernel_ctas(ngroups), kCap, true, &gl);
  if (st == SPX_OK && (classes & 2u))
    st = grid_for(ctx, (const void*)big, kGroupThreads, big_bytes, (ngroups + kGroupThreads - 1) / kGroupThreads, kCap,
                  true, &gb);
  if (st == SPX_OK && (classes & 1u))
    st = grid_for(ctx, (const void*)mid, kMidT, mid_bytes, (ngroups + kMidT - 1) / kMidT, kCap, true, &gm);
  if (st != SPX_OK) return st;
  const int n_all = gs + gl + gb + gm;
  Partial* const p0 = ctx->d_partials;
  Partial* const p1 = ctx->d_partials + n_all;
  const long long* const o = (const long long*)offs;
  cudaStream_t s_big = ctx->stream, s_mid = ctx->stream, s_warp = ctx->stream;
  if (classes != 0u) {
    st = fork_side_streams(ctx);
    if (st != SPX_OK) return st;
    s_mid = ctx->pipe_streams[0];
    s_warp = ctx->pipe_streams[1];
  }
  // the class (1024, 4096] first: it is the long pole of a ragged layout
  if (gb > 0) big<<<gb, kGroupThreads, big_bytes, s_big>>>(s, xk, sj, grad, ngroups, o, lambda_g, nu, p0, xsy, -nu, p1);
  if (gm > 0)
    mid<<<gm, kMidT, mid_bytes, s_mid>>>(s, xk, sj, grad, ngroups, o, lambda_g, nu, p0 + gb, xsy, -nu, p1 + gb);
  lng<<<gl, kGroupThreads, 0, s_warp>>>(s, xk, sj, grad, ngroups, o, lambda_g, nu, classes, p0 + gb + gm, xsy, -nu,
                                        p1 + gb + gm);
  if (gs > 0)
    group_l2_step_kernel<R><<<gs, kGroupThreads, 0, s_warp>>>(s, xsy, xk, sj, grad, ngroups, o, lambda_g, nu, -nu,
                                                               p0 + gb + gm + gl, p1 + gb + gm + gl, true);
  SPX_CUDA(cudaGetLastError());
  ctx->launches += 1 + (gs > 0) + (gb > 0) + (gm > 0);
  *total = n_all;
  if (classes != 0u) return join_side_streams(ctx);
  return SPX_OK;
}

// The norm pass of prox_single_group with q formed from ∇f on the load, on the grid ew_launch gives SolSumSq over the
// same operands (not its own: the instances' register counts, and with them the resident CTAs, may differ), so the
// norm is summed in prox!'s order and s is bit for bit prox!'s
template <class R> static int32_t sol_sumsq_grad_launch(spx_ctx* ctx, const SolSumSqGrad<R>& op, int64_t n, int* nb) {
  constexpr int VECW = 16 / (int)sizeof(R), UNROLL = SolSumSq<R>::UNROLL;
  const bool vec = aligned16(op);
  const long long nvec = vec ? n / VECW : n, tile = (long long)kEwThreads * UNROLL;
  const long long want = std::max(1LL, (nvec + tile - 1) / tile);
  const int per_sm = vec ? ew_blocks_per_sm<VECW, UNROLL, SolSumSq<R>>() : ew_blocks_per_sm<1, UNROLL, SolSumSq<R>>();
  *nb = (int)std::min(want, std::min((long long)ctx->sm_count * per_sm, (long long)kMaxPartials));
  if (vec)
    ew_kernel<VECW, UNROLL, SolSumSqGrad<R>><<<*nb, kEwThreads, 0, ctx->stream>>>(op, n, 0, ctx->d_partials);
  else
    ew_kernel<1, UNROLL, SolSumSqGrad<R>><<<*nb, kEwThreads, 0, ctx->stream>>>(op, n, 0, ctx->d_partials);
  ctx->launches++;
  SPX_CUDA(cudaGetLastError());
  return SPX_OK;
}

// one group spanning the vector: that norm pass, then the scaling pass on step_kernel with xsy and the sums
template <class R>
static int32_t step_single_group(spx_ctx* ctx, int64_t n, R* s, R* xsy, const R* xk, const R* sj, const R* grad,
                                 const R* lambda_g, R nu, double* out3) {
  R lam;
  SPX_CUDA(cudaMemcpyAsync(&lam, lambda_g, sizeof(R), cudaMemcpyDeviceToHost, ctx->stream));
  SolSumSqGrad<R> ss;
  set_in3(ss, xk, sj, grad);
  ss.mnu = -nu;
  int nb = 0;
  int32_t st = sol_sumsq_grad_launch(ctx, ss, n, &nb);
  if (st != SPX_OK) return st;
  st = finalize_partials(ctx, nb, 1, false);  // synchronises: lam has arrived as well
  if (st != SPX_OK) return st;
  const R snorm = (R)std::sqrt(ctx->h_result[0].s2);
  R alpha = R(1) - nu * lam / snorm;  // shiftedGroupNormL2.jl:70-77
  alpha = (alpha != alpha) ? alpha : (alpha > R(0) ? alpha : R(0));
  double v[3];
  st = step_group_scale<R>(ctx, n, s, xsy, xk, sj, grad, nu, alpha, snorm == R(0), v);
  if (st != SPX_OK) return st;
  out3[0] = (double)(R)(double)(lam * (R)std::sqrt(v[0]));
  out3[1] = v[2];
  out3[2] = v[1];
  return SPX_OK;
}

template <class R>
static int32_t step_groupl2(spx_ctx* ctx, int64_t n, R* s, R* xsy, const R* xk, const R* sj, const R* grad,
                            int64_t ngroups, const int64_t* offs, const R* lambda_g, double nu, double* out3) {
  SPX_REQUIRE(n >= 0 && ngroups >= 0, "negative size");
  SPX_STEP_COMMON_CHECKS("spx_step_groupl2", STEP_COMPOSED, ngroups == 0 ? 0 : n, out3);
  SPX_REQUIRE(ngroups == 0 || n == 0 || (sj && offs && lambda_g), "null device vector");
  out3[0] = out3[1] = out3[2] = 0.0;
  if (ngroups == 0 || n == 0) return SPX_OK;
  if (ngroups == 1 && n >= kSingleGroupMin) return step_single_group<R>(ctx, n, s, xsy, xk, sj, grad, lambda_g, (R)nu, out3);
  const spx_ctx::GroupCensus* census = find_census(ctx, offs, ngroups, n);
  int32_t st = SPX_OK;
  if (census && census->classes == 0u) {
    // a validated layout whose groups all have <= 256 elements (the packed warp rounds hold every group)
    int grid = 0;
    st = grid_for(ctx, (const void*)group_l2_step_kernel<R>, kGroupThreads, 0, warp_kernel_ctas(ngroups),
                  kMaxPartials / 2, true, &grid);
    if (st != SPX_OK) return st;
    group_l2_step_kernel<R><<<grid, kGroupThreads, 0, ctx->stream>>>(s, xsy, xk, sj, grad, ngroups, (const long long*)offs,
                                                                    lambda_g, (R)nu, -(R)nu, ctx->d_partials,
                                                                    ctx->d_partials + grid, false);
    ctx->launches++;
    SPX_CUDA(cudaGetLastError());
    st = finalize_partials(ctx, grid, 2, false);
    if (st != SPX_OK) return st;
    out3[0] = ctx->h_result[0].s;
    out3[1] = ctx->h_result[0].s2;
    out3[2] = ctx->h_result[1].s;
    // The flag (folded with max: every rank of a sharded vector sees it) says the layout holds a group of more than 256
    // elements after all -- it was rewritten after validation.  The kernel has written every other group; the
    // long-group kernels take the rest, every class treated as present, and their sums are added to these.
    if (ctx->h_result[0].bad > 0) {
      int total = 0;
      st = launch_step_groupl2<R>(ctx, false, 3u, s, xsy, xk, sj, grad, ngroups, offs, lambda_g, (R)nu, &total);
      if (st == SPX_OK) st = finalize_partials(ctx, total, 2, false);
      if (st != SPX_OK) return st;
      out3[0] += ctx->h_result[0].s;
      out3[1] += ctx->h_result[0].s2;
      out3[2] += ctx->h_result[1].s;
    }
  } else {
    // every other layout: the size classes the census records (all of them for a layout never validated)
    int total = 0;
    st = launch_step_groupl2<R>(ctx, true, census ? census->classes & 3u : 3u, s, xsy, xk, sj, grad, ngroups, offs,
                                lambda_g, (R)nu, &total);
    if (st == SPX_OK) st = finalize_partials(ctx, total, 2, false);
    if (st != SPX_OK) return st;
    out3[0] = ctx->h_result[0].s;
    out3[1] = ctx->h_result[0].s2;
    out3[2] = ctx->h_result[1].s;
  }
  out3[0] = (double)(R)out3[0];  // the reference accumulates ψ in R: one rounding to R
  return SPX_OK;
}

// ---- the solver step of ShiftedGroupNormL2Binf ---------------------------------------------------------------------
//     q = (-ν) ∇f;  prox!(s, ψ, q, ν);  xsy = (xk + sj) + s;  ψ(s) (Inf outside the ball of 1.1Δ);  Σ s²;  Σ ∇f·s
// A uniform layout (the host conditions of prox_group's uniform kernels, and more than one group) runs it in the ONE
// pass of the step form of group_l2binf_uniform_kernel: s is bit for bit what prox! writes.  When the device finds
// offs is not {0, m, 2m, ...} after all, the kernels only raise the redo flag (it travels in the folded slots, so every
// rank of a sharded vector sees it) and the call is redone in the composed form, which every other layout takes at
// once: spx_step_pre, prox! in place with ψ(s) from its value pass, spx_step_post.
template <class R>
static int32_t step_groupl2binf(spx_ctx* ctx, int64_t n, R* s, R* xsy, const R* xk, const R* sj, const R* grad,
                                int64_t ngroups, const int64_t* offs, const R* lambda_g, double nu, double delta,
                                double* out3) {
  SPX_REQUIRE(n >= 0 && ngroups >= 0, "negative size");
  SPX_STEP_COMMON_CHECKS("spx_step_groupl2binf", STEP_COMPOSED, ngroups == 0 ? 0 : n, out3);
  SPX_REQUIRE(ngroups == 0 || n == 0 || (sj && offs && lambda_g), "null device vector");
  out3[0] = out3[1] = out3[2] = 0.0;
  if (ngroups == 0 || n == 0) return SPX_OK;
  const int64_t m = n % ngroups == 0 ? n / ngroups : 0;
  const bool aligned = (((uintptr_t)s | (uintptr_t)xsy | (uintptr_t)xk | (uintptr_t)sj | (uintptr_t)grad) & 15u) == 0;
  if (ngroups > 1 && uniform_binf_candidate(n, m, aligned, nu, delta)) {
    const int64_t nrounds = (n + kRoundElems - 1) / kRoundElems;
    const size_t declined_off = BinfScratch::done_offset(nrounds);
    int32_t st = ensure_scratch(ctx, declined_off + (size_t)nrounds + 256);
    if (st != SPX_OK) return st;
    BinfScratch* const scratch = (BinfScratch*)ctx->d_scratch;
    unsigned* const uniform_flag = &scratch->head.uniform_flag;
    UniformStep<R> step{xsy, -(R)nu, 1.1 * (double)(R)delta, (unsigned char*)ctx->d_scratch + declined_off, 0};
    SPX_CUDA(cudaMemsetAsync(&scratch->head, 0, sizeof(BinfScratch::Head), ctx->stream));
    SPX_CUDA(cudaMemsetAsync(uniform_flag, 1, sizeof(unsigned), ctx->stream));
    SPX_CUDA(cudaMemsetAsync(step.declined, 0, (size_t)nrounds, ctx->stream));
    const int cgrid = (int)std::min<int64_t>((ngroups + 256) / 256, (int64_t)ctx->sm_count * 8);
    group_uniform_check_kernel<<<cgrid, 256, 0, ctx->stream>>>((const long long*)offs, ngroups, m, uniform_flag);
    UDiv<R> by_sigma;
    by_sigma.set((R)nu);
    st = launch_uniform_binf<R, true>(ctx, (int)(m / kEPL), s, xk, sj, grad, ngroups, lambda_g, (R)nu, (R)delta,
                                      by_sigma, uniform_flag, &scratch->head.wl_count, scratch->wl_rounds, &step);
    if (st != SPX_OK) return st;
    ctx->launches += 3;
    SPX_CUDA(cudaGetLastError());
    st = finalize_partials(ctx, step.nblocks, 2, false);
    if (st != SPX_OK) return st;
    if (ctx->h_result[1].bad <= 0) {
      // the reference accumulates ψ in R: one rounding to R here, as value_group_binf
      out3[0] = ctx->h_result[0].bad > 0 ? std::numeric_limits<double>::infinity() : (double)(R)ctx->h_result[0].s;
      out3[1] = ctx->h_result[0].s2;
      out3[2] = ctx->h_result[1].s;
      return SPX_OK;
    }  // else: offs was rewritten after validation and is no longer uniform -- redo the call the long way
  }
  return step_composed<R>(ctx, n, s, xsy, xk, sj, grad, nu, [&](double* psi) {
    return prox_group<R>(ctx, true, n, s, xk, sj, s, ngroups, offs, lambda_g, nu, delta, psi);
  }, out3);
}

}  // namespace spx

using namespace spx;

#ifdef SPX_GROUP_STATS
extern "C" int32_t spx_debug_group_stats(unsigned long long* out2, int reset) {
  cudaMemcpyFromSymbol(out2, g_stat_evals, 8);
  cudaMemcpyFromSymbol(out2 + 1, g_stat_groups, 8);
  cudaMemcpyFromSymbol(out2 + 2, g_stat_big, 24);  // callers pass room for five counters
  if (reset) {
    unsigned long long z = 0;
    cudaMemcpyToSymbol(g_stat_evals, &z, 8);
    cudaMemcpyToSymbol(g_stat_groups, &z, 8);
    unsigned long long z3[3] = {0, 0, 0};
    cudaMemcpyToSymbol(g_stat_big, z3, 24);
  }
  return 0;
}
#endif

// GroupNormL2's constructor checks (groupNormL2.jl:20-23) extended to the device layout: the CSR offsets must start at
// 0, never decrease and end at n -- anything else would make the group kernels read and write out of bounds.
__global__ void __launch_bounds__(256) group_validate_kernel(const long long* __restrict__ offs, long long ngroups,
                                                             long long n, unsigned* bad) {
  bool b = false, mid = false, big = false, lng = false;
  for (long long g = (long long)blockIdx.x * 256 + threadIdx.x; g < ngroups; g += (long long)gridDim.x * 256) {
    const long long lo = offs[g], m = offs[g + 1] - lo;
    b = b || (m < 0) || (lo < 0);
    mid = mid || (m > kMidMin && m <= kBigMin);
    big = big || (m > kBigMin && m <= kBigMax);
    lng = lng || (m > kBigMax);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) b = b || (offs[0] != 0) || (offs[ngroups] != n);
  if (__syncthreads_or(b) && threadIdx.x == 0) bad[0] = 1u;
  // the size classes present (bad[1] bit 0: 257..1024 elements, bit 1: 1025..4096, bit 2: longer), for the census
  const int has_mid = __syncthreads_or(mid), has_big = __syncthreads_or(big), has_lng = __syncthreads_or(lng);
  if (threadIdx.x == 0 && (has_mid || has_big || has_lng))
    atomicOr(&bad[1], (has_mid ? 1u : 0u) | (has_big ? 2u : 0u) | (has_lng ? 4u : 0u));
}
extern "C" int32_t spx_group_validate_offsets(spx_ctx* ctx, int64_t n, int64_t ngroups, const int64_t* offs) {
  SPX_REQUIRE(ctx != nullptr, "null context");
  SPX_REQUIRE(n >= 0 && ngroups >= 0, "negative size");
  SPX_REQUIRE(offs != nullptr, "null offsets");
  DeviceGuard g(ctx->device);
  int32_t st = ensure_scratch(ctx, 4096);
  if (st != SPX_OK) return st;
  unsigned* flag = (unsigned*)ctx->d_scratch;
  SPX_CUDA(cudaMemsetAsync(flag, 0, 2 * sizeof(unsigned), ctx->stream));
  const int grid = (int)std::min<int64_t>((ngroups + 256) / 256, (int64_t)ctx->sm_count * 8);
  group_validate_kernel<<<grid, 256, 0, ctx->stream>>>((const long long*)offs, ngroups, n, flag);
  ctx->launches++;
  unsigned h[2] = {0, 0};
  SPX_CUDA(cudaMemcpyAsync(h, flag, 2 * sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
  SPX_CUDA(cudaStreamSynchronize(ctx->stream));
  // forget whatever was known about this address, then record the layout if it is a valid one
  for (auto& c : ctx->census)
    if (c.offs == (const void*)offs) c = spx_ctx::GroupCensus{};
  if (h[0] != 0) {
    set_error("group offsets must start at 0, be non-decreasing and end at n = %lld", (long long)n);
    return SPX_E_INVALID;
  }
  auto& slot = ctx->census[ctx->census_next];
  ctx->census_next = (ctx->census_next + 1) % (int)(sizeof(ctx->census) / sizeof(ctx->census[0]));
  slot.offs = (const void*)offs;
  slot.ngroups = (long long)ngroups;
  slot.n = (long long)n;
  slot.classes = h[1] & 7u;
  return SPX_OK;
}

#define SPX_DEFINE_GROUP(SUF, R)                                                                                 \
  extern "C" int32_t spx_prox_groupl2_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q, \
                                            int64_t ngroups, const int64_t* offs, const R* lambda_g,             \
                                            double sigma, double* psi_out) {                                     \
    return prox_group<R>(ctx, false, n, y, xk, sj, q, ngroups, offs, lambda_g, sigma, 0.0, psi_out);             \
  }                                                                                                              \
  extern "C" int32_t spx_prox_groupl2binf_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,         \
                                                const R* q, int64_t ngroups, const int64_t* offs,                \
                                                const R* lambda_g, double sigma, double delta,                   \
                                                double* psi_out) {                                               \
    return prox_group<R>(ctx, true, n, y, xk, sj, q, ngroups, offs, lambda_g, sigma, delta, psi_out);            \
  }                                                                                                              \
  extern "C" int32_t spx_value_groupl2_##SUF(spx_ctx* ctx, int64_t n, const R* xk, const R* sj, const R* y,      \
                                             int64_t ngroups, const int64_t* offs, const R* lambda_g,            \
                                             double* out) {                                                      \
    return value_group_binf<R>(ctx, n, xk, sj, y, false, 0.0, ngroups, offs, lambda_g, out);                     \
  }                                                                                                              \
  extern "C" int32_t spx_step_groupl2_##SUF(spx_ctx* ctx, int64_t n, R* s, R* xsy, const R* xk, const R* sj,     \
                                            const R* grad, int64_t ngroups, const int64_t* offs,                 \
                                            const R* lambda_g, double nu, double* out3) {                        \
    return step_groupl2<R>(ctx, n, s, xsy, xk, sj, grad, ngroups, offs, lambda_g, nu, out3);                     \
  }                                                                                                              \
  extern "C" int32_t spx_step_groupl2binf_##SUF(spx_ctx* ctx, int64_t n, R* s, R* xsy, const R* xk, const R* sj, \
                                                const R* grad, int64_t ngroups, const int64_t* offs,             \
                                                const R* lambda_g, double nu, double delta, double* out3) {      \
    return step_groupl2binf<R>(ctx, n, s, xsy, xk, sj, grad, ngroups, offs, lambda_g, nu, delta, out3);          \
  }

SPX_DEFINE_GROUP(f64, double)
SPX_DEFINE_GROUP(f32, float)
