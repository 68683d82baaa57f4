// spx_topr.cu -- ShiftedIndBallL0 / ShiftedIndBallL0BInf prox!: on-device radix-select.
//
// shiftedIndBallL0.jl:54-72, shiftedIndBallL0BInf.jl:73-95.  The reference
// sorts a permutation (`sortperm!(p, y, rev=true, by=abs)`) and zeroes all but
// the first r entries; equal |z| are ordered by ascending index (Base.Perm
// ordering), NaN sorts largest.  Here no permutation exists:
//
//   one thread-block CLUSTER owns one problem.  Each CTA streams its slice of
//   xk, sj, q from HBM exactly once (128-bit loads), keeps z = (xk+sj)+q in
//   registers (16 per thread) and xk+sj in shared memory, and the cluster runs
//   an MSD radix-select (11-bit digits) on the order-preserving integer image
//   of |z|: per-CTA histograms in shared memory (warp-aggregated atomics),
//   summed across the cluster through distributed shared memory.  Ties at the
//   threshold are resolved by an ordered prefix count (lowest index first).
//   y is written once.  HBM traffic = the algorithmic 4R per element.
//
// Problems longer than 8 x 16384 elements take the multi-pass global path at
// the end of this file (z stashed in y, one histogram pass per digit).
#include <cooperative_groups.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "spx_common.cuh"
#include "spx_setup.cuh"

namespace cg = cooperative_groups;

namespace spx {

#ifndef SPX_TR_THREADS
#define SPX_TR_THREADS 1024
#endif
constexpr int kTrThreads = SPX_TR_THREADS;     // 1024 x 64 registers: one CTA per SM (512 x 2 measured slower: 8-CTA clusters)
constexpr int kTrE = 16;                       // elements per thread (registers)
constexpr int kTrChunk = kTrThreads * kTrE;    // 16384 elements per CTA
constexpr int kTrBins = 2048;                  // 11-bit digits
constexpr int kTrBpt = kTrBins / kTrThreads;   // bins per thread when a digit is picked
constexpr int kTrMaxCluster = 8;
constexpr int kTrCandMax = 1024;               // candidates of the threshold bin resolved by direct ranking
constexpr int kPickThreads = 1024;             // single-block digit pick of the global path

#ifdef SPX_TR_TIMING
__device__ unsigned long long g_tr_t[16];
#define TR_T(i)                                          \
  do {                                                   \
    if (threadIdx.x == 0 && blockIdx.x == 0) {           \
      const long long now__ = clock64();                 \
      atomicAdd(&g_tr_t[i], (unsigned long long)(now__ - tr_last)); \
      tr_last = now__;                                   \
    }                                                    \
  } while (0)
#else
#define TR_T(i)
#endif

template <class R> struct KeyTraits;
template <> struct KeyTraits<double> {
  using K = unsigned long long;
  static constexpr int BITS = 63;
  static constexpr int NPASS = 6;
  __device__ static __forceinline__ K key(double z) {
    K k = (K)__double_as_longlong(z) & 0x7fffffffffffffffull;
    return k > 0x7ff0000000000000ull ? 0x7fffffffffffffffull : k;  // every NaN is "largest"
  }
};
template <> struct KeyTraits<float> {
  using K = unsigned int;
  static constexpr int BITS = 31;
  static constexpr int NPASS = 3;
  __device__ static __forceinline__ K key(float z) {
    K k = (K)__float_as_int(z) & 0x7fffffffu;
    return k > 0x7f800000u ? 0x7fffffffu : k;
  }
};
// digit widths, most significant first
__host__ __device__ constexpr int digit_bits(int BITS, int pass) {
  return (BITS - 11 * pass) >= 11 ? 11 : (BITS - 11 * pass);
}

// exclusive prefix sum of one int per thread over the block (ascending thread id);
// `ws` holds 33 ints.  Returns the exclusive prefix; *total = block sum.
template <int THREADS> __device__ __forceinline__ int block_excl_scan(int v, int* ws, int* total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  __syncthreads();  // ws reuse
  if (lane == 31) ws[w] = inc;
  __syncthreads();
  if (w == 0) {
    int s = lane < (THREADS / 32) ? ws[lane] : 0;
    int sinc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, sinc, o);
      if (lane >= o) sinc += t;
    }
    ws[lane] = sinc - s;  // exclusive warp offsets
    if (lane == 31) ws[32] = sinc;
  }
  __syncthreads();
  *total = ws[32];
  return ws[w] + inc - v;
}

// the same scan on 64-bit counts (the histograms of a vector of >= 2^31 elements, or of one summed over 8 GPUs)
template <int THREADS> __device__ __forceinline__ long long block_excl_scan64(long long v, long long* ws, long long* total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  long long inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    long long t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  __syncthreads();  // ws reuse
  if (lane == 31) ws[w] = inc;
  __syncthreads();
  if (w == 0) {
    long long s = lane < (THREADS / 32) ? ws[lane] : 0;
    long long sinc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      long long t = __shfl_up_sync(0xffffffffu, sinc, o);
      if (lane >= o) sinc += t;
    }
    ws[lane] = sinc - s;  // exclusive warp offsets
    if (lane == 31) ws[32] = sinc;
  }
  __syncthreads();
  *total = ws[32];
  return ws[w] + inc - v;
}

struct TrShared {
  unsigned hist[kTrBins];
  unsigned tot[kTrBins];
  int ws[40];
  int sel_bin;
  long long sel_above;
  long long sel_count;
  long long eq_count;  // equal-to-threshold elements in this CTA
  // linear-bin form
  unsigned long long kmax_slot[kTrMaxCluster];  // every CTA's largest key, replicated in every CTA
  unsigned long long cand_key[kTrCandMax];      // CTA 0: keys of the threshold bin
  int cand_idx[kTrCandMax];                     //        and their positions in the problem
  int cand_count;                               // CTA 0
  unsigned long long thr_key;                   // replicated: the r-th largest key ...
  int thr_idx;                                  // ... and the last position kept among its equals
};

template <class R, bool BINF, bool VECLD>
__global__ void __launch_bounds__(kTrThreads, 65536 / (64 * kTrThreads))
    topr_cluster_kernel(R* y, const R* xk, const R* sj, const R* q, long long n, long long r, R delta,
                        long long nprob, const unsigned char* __restrict__ only_flagged) {
  using KT = KeyTraits<R>;
  using K = typename KT::K;
  constexpr int VEC = VECLD ? 16 / (int)sizeof(R) : 1;
  constexpr int ROUNDS = kTrE / VEC;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  TrShared* sh = reinterpret_cast<TrShared*>(smem_raw);
  R* xs_sm = reinterpret_cast<R*>(smem_raw + ((sizeof(TrShared) + 15) / 16) * 16);

  cg::cluster_group cluster = cg::this_cluster();
  const unsigned csize = cluster.num_blocks();
  const unsigned crank = cluster.block_rank();
  const long long ncluster = gridDim.x / csize;
  const long long cid = blockIdx.x / csize;
  const int t = threadIdx.x;
  const int lane = t & 31;

  for (long long prob = cid; prob < nprob; prob += ncluster) {
    if (only_flagged != nullptr && only_flagged[prob] == 0) continue;  // cluster-uniform
    const long long pbase = prob * n;
    const long long cbase = (long long)crank * kTrChunk;  // this CTA's slice of the problem
    long long cnt = n - cbase;
    cnt = cnt < 0 ? 0 : (cnt > kTrChunk ? kTrChunk : cnt);

#ifdef SPX_TR_TIMING
    long long tr_last = clock64();
#endif
    // ---- load: z in registers, xs in shared memory --------------------------
    R z[kTrE];
    unsigned valid = 0;
#pragma unroll
    for (int k = 0; k < ROUNDS; ++k) {
      const long long li = ((long long)k * kTrThreads + t) * VEC;
      if (li < cnt) {  // VECLD => cnt is a multiple of VEC
        Pack<R, VEC> a, b, c;
        ld_stream(xk + pbase + cbase + li, a);
        ld_stream(sj + pbase + cbase + li, b);
        ld_stream(q + pbase + cbase + li, c);
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
          const R xs = a.v[e] + b.v[e];
          z[k * VEC + e] = xs + c.v[e];  // (xk + sj) + q   shiftedIndBallL0.jl:66
          xs_sm[li + e] = xs;
          valid |= 1u << (k * VEC + e);
        }
      } else {
#pragma unroll
        for (int e = 0; e < VEC; ++e) z[k * VEC + e] = R(0);
      }
    }

    __syncthreads();
    TR_T(0);  // load
    // ---- radix select of the r-th largest key ------------------------------
    bool keep_all_bin = true;   // every key whose prefix equals `prefix` is kept
    K prefix = 0;               // selected digits so far
    int shift = KT::BITS;       // bits below the known prefix
    long long need = r;         // rank still to resolve inside the prefix bin
    const bool select = (r > 0) && (r < n);
    if (select) {
      keep_all_bin = false;
      unsigned cand = valid;  // slots whose key still carries the selected prefix
#pragma unroll 1
      for (int pass = 0; pass < KT::NPASS; ++pass) {
        const int width = digit_bits(KT::BITS, pass);
        shift -= width;
        for (int b = t; b < kTrBins; b += kTrThreads) sh->hist[b] = 0;
        __syncthreads();
        const K dmask = (K)((1u << width) - 1u);
        if (__any_sync(0xffffffffu, cand != 0u)) {  // after the first digits most warps hold no candidate
#pragma unroll
          for (int s = 0; s < kTrE; ++s) {
            const bool in = (cand >> s) & 1u;
            if (pass > 0 && !__any_sync(0xffffffffu, in)) continue;
            const unsigned d = in ? (unsigned)((KT::key(z[s]) >> shift) & dmask) : 0xffffffffu;
            const unsigned peers = __match_any_sync(0xffffffffu, d);
            if (in && lane == (__ffs(peers) - 1)) atomicAdd(&sh->hist[d], (unsigned)__popc(peers));
          }
        }
        __syncthreads();
        TR_T(1);  // local histogram
        cluster.sync();  // every CTA's histogram is complete
        TR_T(2);  // cluster sync
        for (int b = t; b < kTrBins; b += kTrThreads) {
          unsigned s = 0;
          for (unsigned rr = 0; rr < csize; ++rr) s += cluster.map_shared_rank(sh->hist, rr)[b];
          sh->tot[b] = s;
        }
        cluster.sync();  // remote reads done before anyone clears its histogram again
        TR_T(3);  // remote sum + sync
        // bins in descending order: thread t owns bins 2047 - kTrBpt t ... 2048 - kTrBpt (t + 1)
        int c[kTrBpt], mine = 0;
#pragma unroll
        for (int j = 0; j < kTrBpt; ++j) {
          c[j] = (int)sh->tot[kTrBins - 1 - kTrBpt * t - j];
          mine += c[j];
        }
        int total;
        long long above = block_excl_scan<kTrThreads>(mine, sh->ws, &total);
#pragma unroll
        for (int j = 0; j < kTrBpt; ++j) {
          if (above < need && need <= above + c[j]) {
            sh->sel_bin = kTrBins - 1 - kTrBpt * t - j;
            sh->sel_above = above;
            sh->sel_count = c[j];
          }
          above += c[j];
        }
        __syncthreads();
        const unsigned sel = (unsigned)sh->sel_bin;
        prefix = (prefix << width) | (K)sel;
        need -= sh->sel_above;
        const long long bin_count = sh->sel_count;
        __syncthreads();
        unsigned keepc = 0;
#pragma unroll
        for (int s = 0; s < kTrE; ++s)
          if (((cand >> s) & 1u) && (unsigned)((KT::key(z[s]) >> shift) & dmask) == sel) keepc |= 1u << s;
        cand = keepc;
        TR_T(4);  // scan + pick
        if (need == bin_count) {  // the whole bin is kept: no finer digit needed
          keep_all_bin = true;
          break;
        }
      }
    }
    // after the loop: element kept iff (key >> shift) > prefix, or == prefix and
    // (keep_all_bin or its rank among the equal elements, in index order, < need)
    const bool keep_everything = !select && r >= n;
    const bool keep_nothing = !select && r <= 0;

    unsigned keepmask = 0;
    if (keep_everything) {
      keepmask = valid;
    } else if (!keep_nothing) {
      unsigned eqmask = 0;
#pragma unroll
      for (int s = 0; s < kTrE; ++s) {
        if ((valid >> s) & 1u) {
          const K kp = KT::key(z[s]) >> shift;
          if (kp > prefix) keepmask |= 1u << s;
          else if (kp == prefix) eqmask |= 1u << s;
        }
      }
      if (keep_all_bin) {
        keepmask |= eqmask;
      } else {
        // ordered tie resolution: equal elements ranked by global index
        int total;
        int mine = __popc(eqmask);
        (void)block_excl_scan<kTrThreads>(mine, sh->ws, &total);
        if (t == 0) sh->eq_count = total;
        cluster.sync();
        long long offset = 0;
        for (unsigned rr = 0; rr < crank; ++rr) offset += *cluster.map_shared_rank(&sh->eq_count, rr);
        cluster.sync();
#pragma unroll 1
        for (int k = 0; k < ROUNDS; ++k) {
          const unsigned m = (eqmask >> (k * VEC)) & ((1u << VEC) - 1u);
          int rtotal;
          long long rank = offset + block_excl_scan<kTrThreads>(__popc(m), sh->ws, &rtotal);
#pragma unroll
          for (int e = 0; e < VEC; ++e) {
            if ((m >> e) & 1u) {
              if (rank < need) keepmask |= 1u << (k * VEC + e);
              ++rank;
            }
          }
          offset += rtotal;
        }
      }
    }

    __syncthreads();
    TR_T(5);  // keep masks / ties
    // ---- write y once -------------------------------------------------------
#pragma unroll
    for (int k = 0; k < ROUNDS; ++k) {
      const long long li = ((long long)k * kTrThreads + t) * VEC;
      if (li < cnt) {
        Pack<R, VEC> o;
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
          const int s = k * VEC + e;
          const R zz = ((keepmask >> s) & 1u) ? z[s] : R(0);
          R v = zz - xs_sm[li + e];  // y .-= xk .+ sj   (:70)
          if (BINF) v = jl_min(jl_max(v, -delta), delta);  // shiftedIndBallL0BInf.jl:91
          o.v[e] = v;
        }
        st_stream(y + pbase + cbase + li, o);
      }
    }
    cluster.sync();  // shared state is reused by the next problem
    TR_T(6);  // write + final sync
  }
}

// ------------------------------------------------------ linear-bin form ---
// The radix digits of an IEEE key are a poor first cut: the top 11 bits are the exponent, which a whole
// problem shares up to a handful of values, so the first pass separates nothing and the select needs ~3
// passes of warp-matched histogram atomics and ~8 cluster barriers.  This form bins |z| LINEARLY between 0
// and the problem's largest magnitude (2048 bins, monotone in |z|, spread over the whole range, so plain
// shared-memory atomics rarely collide): one histogram pass locates the bin holding the r-th largest
// element; that bin holds ~n/2048 elements, which are gathered into CTA 0 and ranked directly (key
// descending, position ascending -- the reference's tie order), giving the exact threshold (key, position).
// Problems it cannot decide cheaply -- a NaN or Inf, all zeros, more than 1024 candidates in the threshold
// bin -- are flagged and left to the radix kernel above, which runs afterwards on the flagged problems only.
template <class R, bool BINF, bool VECLD>
__global__ void __launch_bounds__(kTrThreads, 1)
    topr_cluster_lin_kernel(R* y, const R* xk, const R* sj, const R* q, long long n, long long r, R delta,
                            long long nprob, unsigned char* __restrict__ fallback) {
  using KT = KeyTraits<R>;
  using K = typename KT::K;
  constexpr int VEC = VECLD ? 16 / (int)sizeof(R) : 1;
  constexpr int ROUNDS = kTrE / VEC;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  TrShared* sh = reinterpret_cast<TrShared*>(smem_raw);
  R* xs_sm = reinterpret_cast<R*>(smem_raw + ((sizeof(TrShared) + 15) / 16) * 16);

  cg::cluster_group cluster = cg::this_cluster();
  const unsigned csize = cluster.num_blocks();
  const unsigned crank = cluster.block_rank();
  const long long ncluster = gridDim.x / csize;
  const long long cid = blockIdx.x / csize;
  const int t = threadIdx.x;
  const int lane = t & 31;
  const bool select = (r > 0) && (r < n);
  TrShared* sh0 = cluster.map_shared_rank(sh, 0);

  for (long long prob = cid; prob < nprob; prob += ncluster) {
    const long long pbase = prob * n;
    const long long cbase = (long long)crank * kTrChunk;  // this CTA's slice of the problem
    long long cnt = n - cbase;
    cnt = cnt < 0 ? 0 : (cnt > kTrChunk ? kTrChunk : cnt);

#ifdef SPX_TR_TIMING
    long long tr_last = clock64();
#endif
    // ---- load: z in registers, xs in shared memory --------------------------
    R z[kTrE];
    unsigned valid = 0;
    K kmax = 0;
#pragma unroll
    for (int k = 0; k < ROUNDS; ++k) {
      const long long li = ((long long)k * kTrThreads + t) * VEC;
      if (li < cnt) {  // VECLD => cnt is a multiple of VEC
        Pack<R, VEC> a, b, c;
        ld_stream(xk + pbase + cbase + li, a);
        ld_stream(sj + pbase + cbase + li, b);
        ld_stream(q + pbase + cbase + li, c);
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
          const R xs = a.v[e] + b.v[e];
          z[k * VEC + e] = xs + c.v[e];  // (xk + sj) + q   shiftedIndBallL0.jl:66
          xs_sm[li + e] = xs;
          valid |= 1u << (k * VEC + e);
          const K key = KT::key(z[k * VEC + e]);
          kmax = key > kmax ? key : kmax;
        }
      } else {
#pragma unroll
        for (int e = 0; e < VEC; ++e) z[k * VEC + e] = R(0);
      }
    }
    bool hard = false;
    unsigned keepmask = 0;
    if (!select) {
      keepmask = (r >= n) ? valid : 0u;
    } else {
      __syncthreads();
      TR_T(8);  // load
      // ---- largest magnitude of the problem ---------------------------------
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const K other = __shfl_xor_sync(0xffffffffu, kmax, o);
        kmax = other > kmax ? other : kmax;
      }
      for (int b = t; b < kTrBins; b += kTrThreads) sh->hist[b] = 0;
      if (t == 0) {
        sh->cand_count = 0;
        sh->kmax_slot[crank] = 0;
      }
      __syncthreads();  // also: ws free for reuse
      if (lane == 0) atomicMax(&sh->kmax_slot[crank], (unsigned long long)kmax);
      __syncthreads();
      if (t < (int)csize) cluster.map_shared_rank(sh, t)->kmax_slot[crank] = sh->kmax_slot[crank];
      cluster.sync();
      TR_T(9);  // kmax exchange
      K gmax = 0;
      for (unsigned rr = 0; rr < csize; ++rr) {
        const K v = (K)sh->kmax_slot[rr];
        gmax = v > gmax ? v : gmax;
      }
      // the keys are the bit patterns of |z|: gmax back to a number
      double zmax;
      if (sizeof(R) == 8) zmax = __longlong_as_double((long long)gmax);
      else zmax = (double)__int_as_float((int)gmax);
      const double scale = (double)kTrBins / zmax;
      hard = !(zmax > 0.0) || !(zmax < 1e300) || !(scale < 1e300);  // NaN, Inf, all zero, denormal range
      auto bin_of = [&](R v) -> unsigned {
        const double b = fabs((double)v) * scale;
        const unsigned ub = (unsigned)b;  // b in [0, 2048 (1 + eps)]
        return ub < (unsigned)kTrBins ? ub : (unsigned)kTrBins - 1u;
      };
      long long need = r;
      unsigned sel = 0;
      if (!hard) {
        // ---- one histogram pass ----------------------------------------------
#pragma unroll
        for (int s = 0; s < kTrE; ++s)
          if ((valid >> s) & 1u) atomicAdd(&sh->hist[bin_of(z[s])], 1u);
      }
      __syncthreads();
      TR_T(10);  // histogram
      cluster.sync();  // every CTA's histogram is complete (a hard problem still keeps the barriers aligned)
      if (!hard) {
        for (int b = t; b < kTrBins; b += kTrThreads) {
          unsigned s = 0;
          for (unsigned rr = 0; rr < csize; ++rr) s += cluster.map_shared_rank(sh->hist, rr)[b];
          sh->tot[b] = s;
        }
      }
      cluster.sync();  // remote reads done
      TR_T(11);  // sync + remote sum + sync
      long long bin_count = 0;
      if (!hard) {
        int c[kTrBpt], mine = 0;
#pragma unroll
        for (int j = 0; j < kTrBpt; ++j) {
          c[j] = (int)sh->tot[kTrBins - 1 - kTrBpt * t - j];
          mine += c[j];
        }
        int total;
        long long above = block_excl_scan<kTrThreads>(mine, sh->ws, &total);
#pragma unroll
        for (int j = 0; j < kTrBpt; ++j) {
          if (above < need && need <= above + c[j]) {
            sh->sel_bin = kTrBins - 1 - kTrBpt * t - j;
            sh->sel_above = above;
            sh->sel_count = c[j];
          }
          above += c[j];
        }
        __syncthreads();
        sel = (unsigned)sh->sel_bin;
        need -= sh->sel_above;  // rank inside the threshold bin, 1-based
        bin_count = sh->sel_count;
        hard = bin_count > kTrCandMax;
      }
      TR_T(12);  // scan + pick
      // ---- gather the threshold bin into CTA 0 --------------------------------
      if (!hard) {
#pragma unroll
        for (int k = 0; k < ROUNDS; ++k) {
#pragma unroll
          for (int e = 0; e < VEC; ++e) {
            const int s = k * VEC + e;
            if (((valid >> s) & 1u) && bin_of(z[s]) == sel) {
              const int pos = atomicAdd(&sh0->cand_count, 1);
              sh0->cand_key[pos] = (unsigned long long)KT::key(z[s]);
              sh0->cand_idx[pos] = (int)(cbase + ((long long)k * kTrThreads + t) * VEC + e);
            }
          }
        }
      }
      cluster.sync();
      TR_T(13);  // gather + sync
      if (!hard && crank == 0) {
        // direct ranking: key descending, position ascending; the element of rank `need` is the threshold
        const int C = sh->cand_count;
        for (int ci = t; ci < C; ci += kTrThreads) {
          const unsigned long long mk = sh->cand_key[ci];
          const int mi = sh->cand_idx[ci];
          int rank = 1;
          for (int j = 0; j < C; ++j) {
            const unsigned long long kj = sh->cand_key[j];
            rank += (kj > mk) || (kj == mk && sh->cand_idx[j] < mi);
          }
          if ((long long)rank == need) {
            for (unsigned rr = 0; rr < csize; ++rr) {
              TrShared* dst = cluster.map_shared_rank(sh, rr);
              dst->thr_key = mk;
              dst->thr_idx = mi;
            }
          }
        }
      }
      cluster.sync();
      TR_T(14);  // ranking + sync
      if (!hard) {
        const K tk = (K)sh->thr_key;
        const int ti = sh->thr_idx;
#pragma unroll
        for (int k = 0; k < ROUNDS; ++k) {
#pragma unroll
          for (int e = 0; e < VEC; ++e) {
            const int s = k * VEC + e;
            if ((valid >> s) & 1u) {
              const K key = KT::key(z[s]);
              const int gi = (int)(cbase + ((long long)k * kTrThreads + t) * VEC + e);
              if (key > tk || (key == tk && gi <= ti)) keepmask |= 1u << s;
            }
          }
        }
      }
    }
    if (t == 0 && crank == 0) fallback[prob] = hard ? 1 : 0;

    // ---- write y once (a flagged problem is written by the radix kernel) ------
    if (!hard) {
#pragma unroll
      for (int k = 0; k < ROUNDS; ++k) {
        const long long li = ((long long)k * kTrThreads + t) * VEC;
        if (li < cnt) {
          Pack<R, VEC> o;
#pragma unroll
          for (int e = 0; e < VEC; ++e) {
            const int s = k * VEC + e;
            const R zz = ((keepmask >> s) & 1u) ? z[s] : R(0);
            R v = zz - xs_sm[li + e];  // y .-= xk .+ sj   (:70)
            if (BINF) v = jl_min(jl_max(v, -delta), delta);  // shiftedIndBallL0BInf.jl:91
            o.v[e] = v;
          }
          st_stream(y + pbase + cbase + li, o);
        }
      }
    }
    cluster.sync();  // shared state is reused by the next problem
    TR_T(15);  // keep masks + write + sync
  }
}

// ------------------------------------------- batches of problems: the stream form --
// One CTA per problem, several CTAs per SM, no cluster and no state in registers between phases -- so while one
// CTA of an SM selects, its neighbours stream, which the one-cluster-per-problem form above cannot do (its z pins
// every register of the SM; profiles/r01_topr_lin_phase_timing.txt: 35 % of a problem is select time during which
// the SM pulls nothing from HBM).
//   pass 1  streams xk, sj, q once (3R): writes the DROPPED value of every entry, y_i = clamp(0 - (xk+sj)_i) (1W), and
//           a 16-bit monotone image of |z_i| (the top 16 bits of its Float32 bit pattern: 8 exponent + 7 mantissa
//           bits; NaN -> 0xFFFF) into a per-CTA scratch array that lives in L2 (2 B per element, rewritten for every
//           problem of the CTA);
//   pass 2a re-reads the 16-bit keys (L2), histograms them relative to the problem's largest key (one bin per
//           distinct key value: the 2047 values below the maximum cover 16 binades) and locates the key value t16
//           that holds the r-th largest entry;
//   pass 2b re-reads the keys: an entry with key > t16 is kept whatever the order inside t16 -- its y is rewritten
//           as clamp(z - xs) from the three inputs re-read at that index (~r scattered sectors); entries with
//           key == t16 (a few hundred) are ranked exactly (full key descending, position ascending: the reference's
//           tie order) and the first r - #above of them rewritten the same way.
// HBM traffic = 4R + the scattered re-reads (~r sectors of 32 B per input) + whatever part of the key scratch L2
// writes back.  Problems it cannot decide (NaN / Inf, all zeros, > 1024 candidates, the threshold more than 16
// binades below the maximum) are flagged for the radix kernel above, as in the cluster form.  Not used when y
// aliases an input (pass 1 overwrites y before pass 2 re-reads q at the kept positions).
#ifndef SPX_TS_THREADS
#define SPX_TS_THREADS 256
#endif
#ifndef SPX_TS_MINB
#define SPX_TS_MINB 4
#endif
#ifndef SPX_TS_UNROLL
#define SPX_TS_UNROLL 2
#endif
constexpr int kTsUnroll = SPX_TS_UNROLL;  // 128-bit packets per operand in flight per thread in pass 1
constexpr int kTsCand = 1024;

// L2 residency hints (createpolicy): the streamed operands are marked evict-first, the 16-bit key scratch -- written
// in pass 1 and read twice right after -- evict-last, so the 4R stream does not push the keys out of L2
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void ld_hint(const double* p, Pack<double, 2>& o, uint64_t pol) {
  asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;"
               : "=d"(o.v[0]), "=d"(o.v[1])
               : "l"(p), "l"(pol));
}
__device__ __forceinline__ void ld_hint(const float* p, Pack<float, 4>& o, uint64_t pol) {
  asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
               : "=f"(o.v[0]), "=f"(o.v[1]), "=f"(o.v[2]), "=f"(o.v[3])
               : "l"(p), "l"(pol));
}
__device__ __forceinline__ uint4 ld_keys(const uint4* p, uint64_t pol) {
  uint4 v;
  asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.u32 {%0, %1, %2, %3}, [%4], %5;"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ void st_keys(unsigned* p, unsigned v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.u32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_keys(uint2* p, uint2 v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v2.u32 [%0], {%1, %2}, %3;" ::"l"(p), "r"(v.x), "r"(v.y), "l"(pol) : "memory");
}

template <class R> __device__ __forceinline__ unsigned key16_of(R z) {
  const float f = fabsf((float)z);  // rounding is monotone: the image is non-decreasing in |z|
  const unsigned k = (unsigned)__float_as_int(f) >> 16;
  return (z != z) ? 0xffffu : k;
}

template <bool SMEMKEYS> __device__ __forceinline__ uint4 get_keys(const uint4* p, uint64_t pol) {
  if (SMEMKEYS) return *p;
  return ld_keys(p, pol);
}

template <int THREADS> struct TsShared {
  unsigned hist[kTrBins];
  int ws[40];
  unsigned kmax_w[THREADS / 32];
  int sel_bin;
  long long sel_above, sel_count;
  int cand_count;
  int rewrites;
  int cand_idx[kTsCand];
  unsigned long long cand_key[kTsCand];
};

// The operands the STEP form (spx_step_indballl0) adds: y is s, q is ∇f, and q = mnu ∇f is formed in R on every load.
// a or c, chosen at compile time
template <bool B, class A, class C> __device__ __forceinline__ auto& pick(A& a, C& c) {
  if constexpr (B) return a;
  else return c;
}
template <class R> struct TsStep {
  R* xsy;             // (xk + sj) + s, every element
  R mnu;              // -ν
  double rad;         // BINF: 1.1 Δ in Float64, the ball of ψ(s) (shiftedIndBallL0BInf.jl:44-49)
  Partial* partials;  // slot 0 at [blockIdx.x], slot 1 at [stride + blockIdx.x]
  int stride;
};

// ψ(s), Σ s² and Σ ∇f·s of one entry, added with sign `sg` (+1 for the form written, -1 for the form it replaces).
// The ψ predicates are those of ψ(y): ValueSep (xsy != 0) for the plain type, ValueBinfCount ((sj + s) + xk != 0 and
// |sj + s| > 1.1Δ) for BInf.  The two counts are integers; the violation count leaves in a double slot, exactly.
// One thread's counts of one problem stay within ±2047 (at most 512 entries per thread per pass, plus its candidates),
// so both share one register: cnt = nnz + 4096 viol (the Float64 BInf instances spill with two).
template <class R, bool BINF> struct TsStepAcc {
  double s2 = 0.0, dot = 0.0;
  int cnt = 0;
  __device__ __forceinline__ void add(int sg, R xk, R sj, R xsy, R s, R g, double rad) {
    const double ds = sg > 0 ? (double)s : -(double)s;
    s2 = __fma_rn(ds, (double)s, s2);
    dot = __fma_rn((double)g, ds, dot);
    if (BINF) {
      const R w = sj + s;
      cnt += (fabs((double)w) > rad) ? 4096 * sg : 0;  // w < -rad || w > rad, NaN neither
      cnt += ((w + xk) != R(0)) ? sg : 0;
    } else {
      cnt += (xsy != R(0)) ? sg : 0;
    }
  }
  __device__ __forceinline__ int viol() const { return BINF ? (cnt + 2048) >> 12 : 0; }
  __device__ __forceinline__ int nnz() const { return cnt - 4096 * viol(); }
};

// THREADS x MINB resident threads per SM.  SMEMKEYS: the 16-bit keys of the problem live in (dynamic) shared memory
// -- 2 n bytes, one 1024-thread CTA per SM for n = 65536 -- instead of the L2-resident global scratch (larger n).
// STEP (spx_step_indballl0): y = s and q = ∇f; q = (-ν)∇f is formed in R wherever q was loaded, so keys, selection and
// s are those of prox!(s, ψ, fl(-ν∇f), ν).  Every write of s also writes xsy = (xk + sj) + s.  Pass 1 sums ψ(s),
// Σ s², Σ ∇f·s for the form it wrote; every rewrite of pass 2b adds (new - old).  The candidates of the threshold value
// are rewritten in rank order on a static rank-to-thread map (not in the atomicAdd order of the list), so the sums are
// the same on every call.  A problem's sums go into the CTA's partial slots (slot 0 {ψ count, Σs², flag}, slot 1
// {Σ∇f·s, violations}) after a block fold, unless the problem is hard: then the CTA writes q into its s for the radix
// kernel (run with y = q = s) and topr_step_fixup_kernel writes its xsy and sums.
// Resident CTAs per SM of an instance.  At 64 registers three Float64 STEP forms spill (4 to 36 bytes): the L2-key form
// (n > 102400: global key pointer and cache policies next to the step's sums) and the 256-thread BInf form (the ball
// test next to the clamp).  Those alone run one CTA per SM lower; every other instance keeps its prox! twin's.
template <class R, bool BINF, int THREADS, int MINB, bool SMEMKEYS, bool STEP>
constexpr int ts_min_blocks() {
  return (STEP && sizeof(R) == 8 && (!SMEMKEYS || (BINF && THREADS == 256))) ? MINB - 1 : MINB;
}
template <class R, bool BINF, int THREADS, int MINB, bool SMEMKEYS, bool STEP = false>
__global__ void __launch_bounds__(THREADS, (ts_min_blocks<R, BINF, THREADS, MINB, SMEMKEYS, STEP>()))
    topr_stream_kernel(R* y, const R* xk, const R* sj, const R* q, long long n, long long r, R delta, long long nprob,
                       unsigned short* __restrict__ key_scratch, unsigned char* __restrict__ fallback,
                       TsStep<R> step = TsStep<R>{}) {
  using KT = KeyTraits<R>;
  constexpr int VEC = 16 / (int)sizeof(R);
  constexpr int kTsThreads = THREADS;
  constexpr int kTsBpt = kTrBins / THREADS;
  __shared__ TsShared<THREADS> sh;
  extern __shared__ __align__(16) unsigned char ts_dyn[];
  const int t = threadIdx.x, lane = t & 31;
  const uint64_t pol_stream = l2_policy_evict_first(), pol_keep = l2_policy_evict_last();
  unsigned short* keys = SMEMKEYS ? reinterpret_cast<unsigned short*>(ts_dyn) : key_scratch + (size_t)blockIdx.x * (size_t)n;
  const int nvec = (int)(n / VEC);  // n is a multiple of 8, at most 131072: 32-bit offsets inside a problem
  const int nk8 = (int)(n / 8);
  auto drop = [&](R xs) -> R {
    R v = R(0) - xs;  // a dropped entry: 0 - (xk + sj)   (shiftedIndBallL0.jl:69-70)
    if (BINF) v = jl_min(jl_max(v, -delta), delta);
    return v;
  };
  auto keep = [&](R xs, R z) -> R {
    R v = z - xs;  // a kept entry: z - (xk + sj)   (shiftedIndBallL0.jl:70)
    if (BINF) v = jl_min(jl_max(v, -delta), delta);
    return v;
  };
  auto qof = [&](R qg) -> R {  // STEP: the q plane holds ∇f
    if constexpr (STEP) return step.mnu * qg;
    else return qg;
  };
  auto fix_y = [&](int i, const R* pxk, const R* psj, const R* pq, R* py) {  // rewrite entry i in its kept form
    const R xs = pxk[i] + psj[i];
    py[i] = keep(xs, xs + pq[i]);
  };
  auto unfix_y = [&](int i, const R* pxk, const R* psj, R* py) { py[i] = drop(pxk[i] + psj[i]); };
  // STEP: rewrite entry i of s and xsy in the form `kept`, and add (new - old) to the sums.  The key scan below calls
  // fix / unfix with its original text; in the STEP form they name the wrappers around refix.  Generic lambdas and a
  // compile-time pick rather than `if constexpr` at the call: any branch there changes how the prox! instances compile.
  const R* step_grad = nullptr;  // this problem's ∇f (unfix takes no q operand)
  TsStepAcc<R, BINF> acc;
  auto refix = [&](auto i, bool kept, const R* pxk, const R* psj, const R* pg, R* py, R* pxsy) {
    const R a = pxk[i], b = psj[i], g = pg[i];
    const R xs = a + b;
    const R sk = keep(xs, xs + step.mnu * g), sd = drop(xs);
    const R sn = kept ? sk : sd, so = kept ? sd : sk;
    const R vn = xs + sn;
    py[i] = sn;
    pxsy[i] = vn;
    acc.add(1, a, b, vn, sn, g, step.rad);
    acc.add(-1, a, b, xs + so, so, g, step.rad);
  };
  R* pxsy = nullptr;  // STEP: this problem's xsy
  auto fix_step = [&](auto i, const R* pxk, const R* psj, const R* pg, R* py) { refix(i, true, pxk, psj, pg, py, pxsy); };
  auto unfix_step = [&](auto i, const R* pxk, const R* psj, R* py) { refix(i, false, pxk, psj, step_grad, py, pxsy); };
  auto& fix = pick<STEP>(fix_step, fix_y);
  auto& unfix = pick<STEP>(unfix_step, unfix_y);
  // Pass 1 already writes the KEPT form where the 16-bit key reaches `guess` -- the threshold key of the previous
  // problem of this CTA, which for a batch of like problems is the threshold of this one or its neighbour -- so pass
  // 2b only has to rewrite the entries the guess got wrong plus the unkept ones among the threshold-valued entries,
  // instead of re-reading three operands for every kept entry.  A guess that proves bad (more than r rewrites) is
  // dropped for the next problem.
  unsigned guess = 0x10000u;  // nothing pre-kept
  if constexpr (STEP) {
    if (t == 0) {
      step.partials[blockIdx.x] = Partial{0.0, 0.0, -1};
      step.partials[step.stride + blockIdx.x] = Partial{0.0, 0.0, -1};
    }
  }
  for (long long prob = blockIdx.x; prob < nprob; prob += gridDim.x) {
    const R* pxk = xk + prob * n;
    const R* psj = sj + prob * n;
    const R* pq = q + prob * n;
    R* py = y + prob * n;
    if constexpr (STEP) {
      step_grad = pq;
      pxsy = step.xsy + prob * n;
      acc = TsStepAcc<R, BINF>{};
    }
    // ---- pass 1 -----------------------------------------------------------------------------------------
    unsigned kmax = 0;
    for (int v0 = t; v0 < nvec; v0 += kTsUnroll * kTsThreads) {
      Pack<R, VEC> a[kTsUnroll], b[kTsUnroll], c[kTsUnroll];
#pragma unroll
      for (int u = 0; u < kTsUnroll; ++u) {
        const int v = v0 + u * kTsThreads;
        if (v < nvec) {
          ld_hint(pxk + v * VEC, a[u], pol_stream);
          ld_hint(psj + v * VEC, b[u], pol_stream);
          ld_hint(pq + v * VEC, c[u], pol_stream);
        }
      }
#pragma unroll
      for (int u = 0; u < kTsUnroll; ++u) {
        const int v = v0 + u * kTsThreads;
        if (v < nvec) {
          Pack<R, VEC> o;
          unsigned k16[VEC];
#pragma unroll
          for (int e = 0; e < VEC; ++e) {
            const R xs = a[u].v[e] + b[u].v[e];
            const R z = xs + qof(c[u].v[e]);  // (xk + sj) + q   shiftedIndBallL0.jl:66
            k16[e] = key16_of(z);
            o.v[e] = (k16[e] >= guess) ? keep(xs, z) : drop(xs);
            kmax = k16[e] > kmax ? k16[e] : kmax;
          }
          st_stream(py + v * VEC, o);
          if constexpr (STEP) {
            Pack<R, VEC> w;
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
              w.v[e] = (a[u].v[e] + b[u].v[e]) + o.v[e];
              acc.add(1, a[u].v[e], b[u].v[e], w.v[e], o.v[e], c[u].v[e], step.rad);
            }
            st_stream(pxsy + v * VEC, w);
          }
          if (VEC == 2) {
            const unsigned w = k16[0] | (k16[1] << 16);
            if (SMEMKEYS) reinterpret_cast<unsigned*>(keys)[v] = w;
            else st_keys(reinterpret_cast<unsigned*>(keys) + v, w, pol_keep);
          } else {
            uint2 w;
            w.x = k16[0] | (k16[1] << 16);
            w.y = k16[2 % VEC] | (k16[3 % VEC] << 16);
            if (SMEMKEYS) reinterpret_cast<uint2*>(keys)[v] = w;
            else st_keys(reinterpret_cast<uint2*>(keys) + v, w, pol_keep);
          }
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned other = __shfl_xor_sync(0xffffffffu, kmax, o);
      kmax = other > kmax ? other : kmax;
    }
    if (lane == 0) sh.kmax_w[t >> 5] = kmax;
    for (int b = t; b < kTrBins; b += kTsThreads) sh.hist[b] = 0;
    if (t == 0) {
      sh.cand_count = 0;
      sh.rewrites = 0;
    }
    __syncthreads();  // also orders pass 1's global writes (keys, y) before pass 2's reads / rewrites
    kmax = 0;
#pragma unroll
    for (int w = 0; w < kTsThreads / 32; ++w) kmax = sh.kmax_w[w] > kmax ? sh.kmax_w[w] : kmax;
    const unsigned base16 = kmax > (unsigned)(kTrBins - 1) ? kmax - (unsigned)(kTrBins - 1) : 0u;
    // ---- pass 2a: one bin per key value below the maximum; keys <= base16 are not counted ------------------
    for (int w0 = t - lane; w0 < nk8; w0 += 2 * kTsThreads) {  // warp-uniform trip count: the votes below need every lane
      const int c0 = w0 + lane;
      uint4 wv[2];
#pragma unroll
      for (int u = 0; u < 2; ++u)
        wv[u] = (c0 + u * kTsThreads < nk8) ? get_keys<SMEMKEYS>(reinterpret_cast<const uint4*>(keys) + c0 + u * kTsThreads, pol_keep)
                                            : make_uint4(0u, 0u, 0u, 0u);  // key 0 is never counted
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const unsigned ww[4] = {wv[u].x, wv[u].y, wv[u].z, wv[u].w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const unsigned k = (ww[j >> 1] >> ((j & 1) * 16)) & 0xffffu;
          const bool cnt = k > base16;
          // a warp whose lanes all hit one bin (constant data, massive ties) adds once
          const unsigned k0 = __shfl_sync(0xffffffffu, k, 0);
          if (__all_sync(0xffffffffu, k == k0)) {
            if (lane == 0 && cnt) atomicAdd(&sh.hist[k - base16], 32u);
          } else if (cnt) {
            atomicAdd(&sh.hist[k - base16], 1u);
          }
        }
      }
    }
    __syncthreads();
    // ---- pick the key value holding the r-th largest entry ----------------------------------------------
    bool hard;
    unsigned t16 = 0;
    long long need = 0;
    {
      int c[kTsBpt], mine = 0;
#pragma unroll
      for (int j = 0; j < kTsBpt; ++j) {
        c[j] = (int)sh.hist[kTrBins - 1 - kTsBpt * t - j];
        mine += c[j];
      }
      if (t == 0) sh.sel_bin = 0;
      int total;
      long long above = block_excl_scan<kTsThreads>(mine, sh.ws, &total);
#pragma unroll
      for (int j = 0; j < kTsBpt; ++j) {
        const int bin = kTrBins - 1 - kTsBpt * t - j;
        if (bin > 0 && above < r && r <= above + c[j]) {
          sh.sel_bin = bin;
          sh.sel_above = above;
          sh.sel_count = c[j];
        }
        above += c[j];
      }
      __syncthreads();
      const int sel = sh.sel_bin;
      // bin 0 (everything 16 binades below the maximum, zeros, the all-equal-to-zero problem), a NaN / Inf
      // maximum, or a crowded threshold value: left to the radix kernel
      hard = (sel == 0) || (kmax >= 0x7f80u) || (sh.sel_count > (long long)kTsCand);
      t16 = base16 + (unsigned)sel;
      need = r - sh.sel_above;  // rank inside the threshold value, 1-based
    }
    if (t == 0) fallback[prob] = hard ? 1 : 0;
    if (!hard) {
      // ---- pass 2b: entries pass 1 wrote in the wrong form rewritten, threshold-valued entries listed -----------
      int nrewrite = 0;
      for (int c8 = t; c8 < nk8; c8 += kTsThreads) {
        const uint4 w = get_keys<SMEMKEYS>(reinterpret_cast<const uint4*>(keys) + c8, pol_stream);
        const unsigned ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const unsigned k = (ww[j >> 1] >> ((j & 1) * 16)) & 0xffffu;
          const int i = c8 * 8 + j;
          if (k == t16) {
            const int pos = atomicAdd(&sh.cand_count, 1);
            if (pos < kTsCand) sh.cand_idx[pos] = i;
          } else if ((k > t16) != (k >= guess)) {  // pass 1 wrote the other form
            if (k > t16) fix(i, pxk, psj, pq, py);
            else unfix(i, pxk, psj, py);
            ++nrewrite;
          }
        }
      }
      __syncthreads();
      const int C = sh.cand_count < kTsCand ? sh.cand_count : kTsCand;  // == sel_count <= kTsCand
      for (int ci = t; ci < C; ci += kTsThreads) {
        const int i = sh.cand_idx[ci];
        const R z = (pxk[i] + psj[i]) + qof(pq[i]);
        sh.cand_key[ci] = (unsigned long long)KT::key(z);
      }
      __syncthreads();
      // direct ranking: key descending, position ascending; the first `need` are kept
      for (int ci = t; ci < C; ci += kTsThreads) {
        const unsigned long long mk = sh.cand_key[ci];
        const int mi = sh.cand_idx[ci];
        int rank = 1;
        for (int j = 0; j < C; ++j) {
          const unsigned long long kj = sh.cand_key[j];
          rank += (kj > mk) || (kj == mk && sh.cand_idx[j] < mi);
        }
        if constexpr (STEP) {
          reinterpret_cast<int*>(sh.hist)[rank - 1] = mi;  // ranks are 1..C, each once; hist is free after the pick
        } else {
          const bool kept = (long long)rank <= need;
          if (kept != (t16 >= guess)) {
            if (kept) fix(mi, pxk, psj, pq, py);
            else unfix(mi, pxk, psj, py);
          }
        }
      }
      if constexpr (STEP) {
        __syncthreads();
        for (int rk = t; rk < C; rk += kTsThreads) {  // the candidate of rank rk + 1, on a static map
          const bool kept = (long long)rk < need;
          if (kept != (t16 >= guess)) refix(reinterpret_cast<const int*>(sh.hist)[rk], kept, pxk, psj, pq, py, pxsy);
        }
      }
      if (nrewrite) atomicAdd(&sh.rewrites, nrewrite);
    }
    if constexpr (STEP) {
      if (hard) {  // q into s for the radix kernel, which runs on the flagged problems with y = q = s
        for (int v = t; v < nvec; v += kTsThreads) {
          Pack<R, VEC> g;
          ld_stream(pq + v * VEC, g);
#pragma unroll
          for (int e = 0; e < VEC; ++e) g.v[e] = step.mnu * g.v[e];
          st_stream(py + v * VEC, g);
        }
      } else {  // block-uniform
        Partial p0, p1;
        p0.s = (double)acc.nnz();
        p0.s2 = acc.s2;
        p0.bad = -1;
        p1.s = acc.dot;
        p1.s2 = (double)acc.viol();
        p1.bad = -1;
        p0 = block_fold<kTsThreads>(p0);
        p1 = block_fold<kTsThreads>(p1);
        if (t == 0) {  // the CTA owns its slots: plain read-modify-write, problems in a fixed order
          Partial* s0 = step.partials + blockIdx.x;
          Partial* s1 = step.partials + step.stride + blockIdx.x;
          s0->s += p0.s;
          s0->s2 += p0.s2;
          s1->s += p1.s;
          s1->s2 += p1.s2;
          s0->bad = s1->s2 > 0.0 ? 1 : -1;  // BINF: an entry of sj + s outside the ball (the exact count)
        }
      }
    }
    __syncthreads();  // shared state (and the key scratch) is reused by the next problem
    guess = (!hard && (long long)sh.rewrites <= r) ? t16 : 0x10000u;
    __syncthreads();
  }
}

// The step's problems that the stream kernel flagged and the radix kernel then solved in place: xsy = (xk + sj) + s and
// the sums of the STEP form, into partial slots of their own.  A fixed grid walks the problems on a static map and
// skips the unflagged ones, so the sums come out the same on every call; with no flagged problem it only reads flags.
constexpr int kFixThreads = 256;
template <class R, bool BINF>
__global__ void __launch_bounds__(kFixThreads)
    topr_step_fixup_kernel(const R* s, R* xsy, const R* xk, const R* sj, const R* grad, long long n, long long nprob,
                           double rad, const unsigned char* __restrict__ flagged, Partial* partials, int stride) {
  TsStepAcc<R, BINF> acc;  // its packed count is emptied after every problem (at most n / 256 <= 512 entries)
  double nnz = 0.0, viol = 0.0;
  for (long long prob = blockIdx.x; prob < nprob; prob += gridDim.x) {
    if (flagged[prob] == 0) continue;  // block-uniform
    const long long b = prob * n;
    for (long long i = b + threadIdx.x; i < b + n; i += kFixThreads) {
      const R a = xk[i], c = sj[i], v = s[i];
      const R w = (a + c) + v;
      xsy[i] = w;
      acc.add(1, a, c, w, v, grad[i], rad);
    }
    nnz += (double)acc.nnz();
    viol += (double)acc.viol();
    acc.cnt = 0;
  }
  Partial p0, p1;
  p0.s = nnz;
  p0.s2 = acc.s2;
  p0.bad = viol > 0.0 ? 1 : -1;
  p1.s = acc.dot;
  p1.s2 = viol;
  p1.bad = -1;
  p0 = block_fold<kFixThreads>(p0);
  p1 = block_fold<kFixThreads>(p1);
  if (threadIdx.x == 0) {
    partials[blockIdx.x] = p0;
    partials[stride + blockIdx.x] = p1;
  }
}

// ------------------------------------------------- global multi-pass path ---
// For one long vector: z is stashed in y (3R + 1W), every further digit costs
// one read of y (until the selected bin is down to the elements it keeps: two such passes on random Float64 data), the
// last pass reads y, xk, sj and writes y; the tie ranks of the last pass come from per-warp slices (no block barrier).
struct GlobalSel {
  unsigned long long hist[kTrBins];  // 64-bit: the sharded form sums the histograms of every GPU
  unsigned long long prefix;
  long long need;
  int shift;
  int done;          // keep_all_bin reached
  long long eq_total;
  long long eq_base;  // threshold-equal elements on lower-ranked shards (sharded form)
};

template <class R>
__global__ void __launch_bounds__(256) topr_g_stash(R* y, const R* xk, const R* sj, const R* q, long long n,
                                                    GlobalSel* st) {
  using KT = KeyTraits<R>;
  __shared__ unsigned h[kTrBins];
  for (int b = threadIdx.x; b < kTrBins; b += 256) h[b] = 0;
  __syncthreads();
  const int width = digit_bits(KT::BITS, 0);
  const int shift = KT::BITS - width;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const R z = (xk[i] + sj[i]) + q[i];
    y[i] = z;
    atomicAdd(&h[(unsigned)(KT::key(z) >> shift)], 1u);
  }
  __syncthreads();
  for (int b = threadIdx.x; b < kTrBins; b += 256)
    if (h[b]) atomicAdd(&st->hist[b], (unsigned long long)h[b]);
}

template <class R>
__global__ void __launch_bounds__(256) topr_g_hist(const R* y, long long n, int pass, GlobalSel* st) {
  using KT = KeyTraits<R>;
  using K = typename KT::K;
  __shared__ unsigned h[kTrBins];
  if (st->done) return;
  for (int b = threadIdx.x; b < kTrBins; b += 256) h[b] = 0;
  __syncthreads();
  const int width = digit_bits(KT::BITS, pass);
  const int hi_shift = st->shift;
  const int shift = hi_shift - width;
  const K prefix = (K)st->prefix;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const K key = KT::key(y[i]);
    if ((key >> hi_shift) == prefix) atomicAdd(&h[(unsigned)((key >> shift) & (K)((1u << width) - 1u))], 1u);
  }
  __syncthreads();
  for (int b = threadIdx.x; b < kTrBins; b += 256)
    if (h[b]) atomicAdd(&st->hist[b], (unsigned long long)h[b]);
}

// single block: pick the digit, update the selection state, clear the histogram
template <class R>
__global__ void __launch_bounds__(kPickThreads) topr_g_pick(int pass, GlobalSel* st) {
  using KT = KeyTraits<R>;
  __shared__ long long ws[40];
  __shared__ int sel_bin;
  __shared__ long long sel_above, sel_count;
  if (st->done) return;
  const int t = threadIdx.x;
  const int width = digit_bits(KT::BITS, pass);
  const int b0 = kTrBins - 1 - 2 * t, b1 = b0 - 1;
  const long long c0 = (long long)st->hist[b0], c1 = (long long)st->hist[b1];
  // 64-bit scan: a bin of the first digit can hold every element of the vector (n_global >= 2^31 for a Float32
  // vector on one B200, or for the histogram summed over the GPUs of a box)
  long long total;
  const long long above = block_excl_scan64<kPickThreads>(c0 + c1, ws, &total);
  const long long need = st->need;
  if (above < need && need <= above + c0) {
    sel_bin = b0; sel_above = above; sel_count = c0;
  } else if (above + c0 < need && need <= above + c0 + c1) {
    sel_bin = b1; sel_above = above + c0; sel_count = c1;
  }
  __syncthreads();
  st->hist[b0] = 0;
  st->hist[b1] = 0;
  if (t == 0) {
    st->prefix = (st->prefix << width) | (unsigned long long)sel_bin;
    st->need = need - sel_above;
    st->shift -= width;
    if (st->need == sel_count) st->done = 1;
  }
}

// Tie ranks (lowest index first among the threshold-equal entries) need the number of such entries in front of every
// element.  The vector is cut into one contiguous slice per WARP of the final pass (per_slice elements, a multiple of
// 128): this kernel counts the threshold-equal entries of each slice, topr_g_scan turns the counts into exclusive
// prefixes, and the final pass ranks inside a slice with ballots only -- no block barrier anywhere in it.
template <class R>
__global__ void __launch_bounds__(256) topr_g_eqcount(const R* y, long long n, long long per_slice,
                                                      const GlobalSel* st, long long* slice_eq) {
  using KT = KeyTraits<R>;
  using K = typename KT::K;
  const int lane = threadIdx.x & 31;
  const long long slice = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (st->done) {
    if (lane == 0) slice_eq[slice] = 0;
    return;
  }
  const long long b = slice * per_slice;
  const long long e = b + per_slice < n ? b + per_slice : n;
  const K prefix = (K)st->prefix;
  const int shift = st->shift;
  long long c = 0;
#pragma unroll 4
  for (long long i = b + lane; i < e; i += 32) c += (KT::key(y[i]) >> shift) == prefix;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane == 0) slice_eq[slice] = c;
}
// exclusive prefix sums of the slice counts (one block of 1024 threads, consecutive runs of slices per thread)
__global__ void __launch_bounds__(1024) topr_g_scan(long long* slice_eq, int nslices, GlobalSel* st) {
  __shared__ long long ws[40];
  const int per = (nslices + 1023) / 1024;
  const int b = threadIdx.x * per, e = min(b + per, nslices);
  long long local = 0;
  for (int i = b; i < e; ++i) local += slice_eq[i];
  long long total;
  long long run = block_excl_scan64<1024>(local, ws, &total);
  for (int i = b; i < e; ++i) {
    const long long c = slice_eq[i];
    slice_eq[i] = run;
    run += c;
  }
  if (threadIdx.x == 0) st->eq_total = total;
}

// phase 0: slots[rr] = (rr == rank) ? this shard's threshold-equal count : 0;  phase 1 (after the sum over ranks):
// eq_base = the counts of the lower-ranked shards
__global__ void topr_g_rank_slot(long long* slots, int world, int rank, GlobalSel* st, int phase) {
  if (phase == 0) {
    for (int rr = threadIdx.x; rr < world; rr += blockDim.x) slots[rr] = rr == rank ? st->eq_total : 0;
  } else if (threadIdx.x == 0) {
    long long base = 0;
    for (int rr = 0; rr < rank; ++rr) base += slots[rr];
    st->eq_base = base;
  }
}

template <class R, bool BINF>
__global__ void __launch_bounds__(256) topr_g_final(R* y, const R* xk, const R* sj, long long n, long long per_slice,
                                                    const GlobalSel* st, const long long* slice_eq, R delta,
                                                    int mode /*0 select, 1 keep all, 2 keep none*/) {
  using KT = KeyTraits<R>;
  using K = typename KT::K;
  constexpr int U = 4;  // 32-element chunks per trip: 3 U independent loads per lane in flight
  const int lane = threadIdx.x & 31;
  const long long slice = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const long long b = slice * per_slice;
  const long long e = b + per_slice < n ? b + per_slice : n;
  const K prefix = (K)st->prefix;
  const int shift = st->shift;
  const bool all_bin = st->done != 0;
  const long long need = st->need;
  long long run = (mode == 0 && !all_bin) ? st->eq_base + slice_eq[slice] : 0;  // threshold-equal entries in front
  for (long long base = b; base < e; base += 32 * U) {
    R z[U], xs[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = base + u * 32 + lane;
      z[u] = R(0);
      xs[u] = R(0);
      if (i < e) {
        z[u] = y[i];
        xs[u] = xk[i] + sj[i];
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = base + u * 32 + lane;
      bool keep = mode == 1;
      if (mode == 0) {
        const K kp = KT::key(z[u]) >> shift;
        const bool eq = i < e && kp == prefix;
        keep = kp > prefix;
        if (all_bin) {
          keep = keep || eq;
        } else {  // lowest index first: rank among the threshold-equal entries of the shard(s)
          const unsigned bal = __ballot_sync(0xffffffffu, eq);
          const long long rank = run + __popc(bal & ((1u << lane) - 1u));
          keep = keep || (eq && rank < need);
          run += __popc(bal);
        }
      }
      if (i < e) {
        R v = (keep ? z[u] : R(0)) - xs[u];
        if (BINF) v = jl_min(jl_max(v, -delta), delta);
        y[i] = v;
      }
    }
  }
}

// One vector on one GPU (reduce == nullptr), or this GPU's contiguous shard of a vector spread over
// `world` GPUs in rank order: the histogram of every digit is summed over the shards through the caller's
// all-reduce (SURVEY.md §8e: one exchange per radix digit), every rank picks the same digit, and the
// lowest-index tie rule continues across shards through the count of threshold-equal elements on the
// lower-ranked shards.
template <class R>
static int32_t topr_global(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q, int64_t r, bool binf,
                           R delta, int64_t n_global = -1, int rank = 0, int world = 1,
                           spx_allreduce_sum_fn reduce = nullptr, void* user = nullptr) {
  using KT = KeyTraits<R>;
  if (n_global < 0) n_global = n;
  const int nblk = ctx->sm_count * 8;
  const int nslices = nblk * 8;  // one contiguous slice of the vector per warp of the counting / final passes
  int32_t stt = ensure_scratch(ctx, sizeof(GlobalSel) + sizeof(long long) * (size_t)(nslices + 1 + 64));
  if (stt != SPX_OK) return stt;
  GlobalSel* st = (GlobalSel*)ctx->d_scratch;
  long long* block_eq = (long long*)((char*)ctx->d_scratch + sizeof(GlobalSel));
  GlobalSel init;
  memset(&init, 0, sizeof(init));
  init.need = r;
  init.shift = KT::BITS;
  SPX_CUDA(cudaMemcpyAsync(st, &init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
  const int mode = (r >= n_global) ? 1 : (r <= 0 ? 2 : 0);
  // sum the histogram over the shards (counts are exact in Float64 up to 2^53)
  std::vector<unsigned long long> hh;
  std::vector<double> hd;
  const bool lib_comm = !reduce && world > 1;  // the communicator of the context: all-reduce on the device
  auto reduce_hist = [&]() -> int32_t {
    if (lib_comm) return comm_allreduce_raw(ctx, st->hist, kTrBins, kNcclUint64, kNcclSum);
    if (!reduce) return SPX_OK;
    hh.resize(kTrBins);
    hd.resize(kTrBins);
    SPX_CUDA(cudaMemcpyAsync(hh.data(), st->hist, sizeof(unsigned long long) * kTrBins, cudaMemcpyDeviceToHost,
                             ctx->stream));
    SPX_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int b = 0; b < kTrBins; ++b) hd[b] = (double)hh[b];
    int32_t st2 = reduce(user, hd.data(), kTrBins);
    if (st2 != SPX_OK) {
      set_error("spx_prox_indballl0_sharded: all-reduce callback failed (%d)", (int)st2);
      return st2;
    }
    for (int b = 0; b < kTrBins; ++b) hh[b] = (unsigned long long)hd[b];
    SPX_CUDA(cudaMemcpyAsync(st->hist, hh.data(), sizeof(unsigned long long) * kTrBins, cudaMemcpyHostToDevice,
                             ctx->stream));
    return SPX_OK;
  };
  if (n > 0) {
    topr_g_stash<R><<<nblk, 256, 0, ctx->stream>>>(y, xk, sj, q, n, st);
    ctx->launches++;
  }
  const long long per_slice = ((n + nslices - 1) / nslices + 127) / 128 * 128;
  if (mode == 0) {
    for (int pass = 0; pass < KT::NPASS; ++pass) {
      if (pass > 0 && n > 0) {
        topr_g_hist<R><<<nblk, 256, 0, ctx->stream>>>(y, n, pass, st);
        ctx->launches++;
      }
      stt = reduce_hist();
      if (stt != SPX_OK) return stt;
      topr_g_pick<R><<<1, kPickThreads, 0, ctx->stream>>>(pass, st);
      ctx->launches++;
    }
    topr_g_eqcount<R><<<nblk, 256, 0, ctx->stream>>>(y, n, per_slice, st, block_eq);
    topr_g_scan<<<1, 1024, 0, ctx->stream>>>(block_eq, nslices, st);
    ctx->launches += 2;
    if (lib_comm) {
      // exclusive prefix over ranks of the threshold-equal counts, on the device: one slot per rank, summed
      long long* slots = block_eq + nslices + 1;
      topr_g_rank_slot<<<1, 64, 0, ctx->stream>>>(slots, world, rank, st, 0);
      int32_t st2 = comm_allreduce_raw(ctx, slots, (size_t)world, kNcclInt64, kNcclSum);
      if (st2 != SPX_OK) return st2;
      topr_g_rank_slot<<<1, 64, 0, ctx->stream>>>(slots, world, rank, st, 1);
      ctx->launches += 2;
    } else if (reduce && world > 1) {
      // exclusive prefix over ranks of the threshold-equal counts: all-reduce a vector with one slot per rank
      long long eq_total = 0;
      SPX_CUDA(cudaMemcpyAsync(&eq_total, &st->eq_total, sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
      SPX_CUDA(cudaStreamSynchronize(ctx->stream));
      std::vector<double> slots((size_t)world, 0.0);
      slots[(size_t)rank] = (double)eq_total;
      int32_t st2 = reduce(user, slots.data(), world);
      if (st2 != SPX_OK) {
        set_error("spx_prox_indballl0_sharded: all-reduce callback failed (%d)", (int)st2);
        return st2;
      }
      long long base = 0;
      for (int rr = 0; rr < rank; ++rr) base += (long long)slots[(size_t)rr];
      SPX_CUDA(cudaMemcpyAsync(&st->eq_base, &base, sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
      SPX_CUDA(cudaStreamSynchronize(ctx->stream));  // `base` lives on this stack frame
    }
  }
  if (n > 0) {
    if (binf)
      topr_g_final<R, true><<<nblk, 256, 0, ctx->stream>>>(y, xk, sj, n, per_slice, st, block_eq, delta, mode);
    else
      topr_g_final<R, false><<<nblk, 256, 0, ctx->stream>>>(y, xk, sj, n, per_slice, st, block_eq, delta, mode);
    ctx->launches++;
  }
  SPX_CUDA(cudaGetLastError());
  return SPX_OK;
}

template <class Kern>
static int32_t cluster_grid(spx_ctx* ctx, Kern kern, int csize, size_t smem, int64_t nprob, cudaLaunchConfig_t* cfg,
                            cudaLaunchAttribute* attr) {
  SPX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = csize;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg->blockDim = dim3(kTrThreads);
  cfg->dynamicSmemBytes = smem;
  cfg->stream = ctx->stream;
  cfg->attrs = attr;
  cfg->numAttrs = 1;
  cfg->gridDim = dim3(csize);
  int max_clusters = 0;
  cudaError_t e = cudaOccupancyMaxActiveClusters(&max_clusters, kern, cfg);
  if (e != cudaSuccess || max_clusters < 1) max_clusters = ctx->sm_count / csize;
  if (max_clusters < 1) max_clusters = 1;
  long long nclusters = nprob < max_clusters ? nprob : max_clusters;
  cfg->gridDim = dim3((unsigned)(nclusters * csize));
  return SPX_OK;
}

template <class R, bool BINF, bool VECLD>
static int32_t topr_cluster_launch(spx_ctx* ctx, int64_t nprob, int64_t n, R* y, const R* xk, const R* sj, const R* q,
                                   int64_t r, R delta) {
  int csize = 1;
  while ((long long)csize * kTrChunk < n) csize <<= 1;
  const size_t smem = ((sizeof(TrShared) + 15) / 16) * 16 + sizeof(R) * (size_t)kTrChunk;
  int32_t st = ensure_scratch(ctx, (size_t)nprob + 4096);
  if (st != SPX_OK) return st;
  unsigned char* flags = (unsigned char*)ctx->d_scratch + 4096;  // the first 4 KiB belong to the reductions
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  {  // linear-bin select: decides every ordinary problem
    auto kern = topr_cluster_lin_kernel<R, BINF, VECLD>;
    st = cluster_grid(ctx, kern, csize, smem, nprob, &cfg, attr);
    if (st != SPX_OK) return st;
    SPX_CUDA(cudaLaunchKernelEx(&cfg, kern, y, xk, sj, q, (long long)n, (long long)r, delta, (long long)nprob, flags));
    ctx->launches++;
  }
  {  // radix select on the problems it flagged (NaN / Inf / all-zero / crowded threshold bin)
    auto kern = topr_cluster_kernel<R, BINF, VECLD>;
    st = cluster_grid(ctx, kern, csize, smem, nprob, &cfg, attr);
    if (st != SPX_OK) return st;
    SPX_CUDA(cudaLaunchKernelEx(&cfg, kern, y, xk, sj, q, (long long)n, (long long)r, delta, (long long)nprob,
                                (const unsigned char*)flags));
    ctx->launches++;
  }
  return SPX_OK;
}

// STEP (spx_step_indballl0): y = s, q = ∇f, and `step` carries xsy, -ν, the ball and the partial slots; the radix kernel
// then runs with q = s, and *step_grid returns the stream grid (the fixup kernel's slots follow it).
template <class R, bool BINF, bool STEP = false>
static int32_t topr_stream_launch(spx_ctx* ctx, int64_t nprob, int64_t n, R* y, const R* xk, const R* sj, const R* q,
                                  int64_t r, R delta, TsStep<R> step = TsStep<R>{}, int* step_grid = nullptr) {
  const size_t flags_bytes = ((size_t)nprob + 255) & ~(size_t)255;
  const size_t key_bytes = (size_t)n * sizeof(unsigned short);
  // keys in shared memory while 2 n bytes fit next to the static state of a CTA: one 1024-thread CTA per SM above
  // 72 KiB of keys, two 512-thread CTAs down to 36 KiB, four 256-thread CTAs below
  const bool smem_keys = key_bytes <= 200 * 1024;
  int32_t st = SPX_OK;
  unsigned char* flags = nullptr;
  auto go = [&](auto kern, int threads, size_t dyn, bool scratch_keys) -> int32_t {
    if (dyn > 0) SPX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    int per_sm = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, dyn) != cudaSuccess || per_sm < 1) per_sm = 1;
    const int64_t grid = std::min<int64_t>(nprob, (int64_t)ctx->sm_count * per_sm);
    int32_t s2 = ensure_scratch(ctx, 4096 + flags_bytes + (scratch_keys ? (size_t)grid * key_bytes : 0));
    if (s2 != SPX_OK) return s2;
    flags = (unsigned char*)ctx->d_scratch + 4096;  // the first 4 KiB belong to the reductions
    unsigned short* keys = (unsigned short*)((char*)ctx->d_scratch + 4096 + flags_bytes);
    if constexpr (STEP) {
      step.stride = (int)grid + ctx->sm_count;  // the fixup kernel's sm_count CTAs follow the stream grid
      *step_grid = (int)grid;
    }
    kern<<<(unsigned)grid, threads, dyn, ctx->stream>>>(y, xk, sj, q, (long long)n, (long long)r, delta, (long long)nprob,
                                                        keys, flags, step);
    ctx->launches++;
    SPX_CUDA(cudaGetLastError());
    return SPX_OK;
  };
  if (!smem_keys) st = go(topr_stream_kernel<R, BINF, 512, 2, false, STEP>, 512, 0, true);
  else if (key_bytes > 72 * 1024) st = go(topr_stream_kernel<R, BINF, 1024, 1, true, STEP>, 1024, key_bytes, false);
  else if (key_bytes > 36 * 1024) st = go(topr_stream_kernel<R, BINF, 512, 2, true, STEP>, 512, key_bytes, false);
  else st = go(topr_stream_kernel<R, BINF, 256, 4, true, STEP>, 256, key_bytes, false);
  if (st != SPX_OK) return st;
  // radix select on the problems it flagged (NaN / Inf / all-zero / crowded threshold value)
  int csize = 1;
  while ((long long)csize * kTrChunk < n) csize <<= 1;
  const size_t smem = ((sizeof(TrShared) + 15) / 16) * 16 + sizeof(R) * (size_t)kTrChunk;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  auto rk = topr_cluster_kernel<R, BINF, true>;
  st = cluster_grid(ctx, rk, csize, smem, nprob, &cfg, attr);
  if (st != SPX_OK) return st;
  SPX_CUDA(cudaLaunchKernelEx(&cfg, rk, y, xk, sj, STEP ? (const R*)y : q, (long long)n, (long long)r, delta,
                              (long long)nprob, (const unsigned char*)flags));
  ctx->launches++;
  if constexpr (STEP) {
    topr_step_fixup_kernel<R, BINF><<<ctx->sm_count, kFixThreads, 0, ctx->stream>>>(
        y, step.xsy, xk, sj, q, (long long)n, (long long)nprob, step.rad, flags, step.partials + *step_grid,
        step.stride);
    ctx->launches++;
    SPX_CUDA(cudaGetLastError());
  }
  return SPX_OK;
}

// The host conditions of the stream form (batches of problems: one CTA per problem), shared by prox! and the step:
// 16-byte aligned vectors, n a multiple of 8 in [4096, the cluster capacity], 0 < r < n, at least two problems per SM,
// and no output overlapping an input (pass 1 writes y before pass 2b re-reads the inputs at the kept positions).
template <class R>
static bool topr_stream_ok(const spx_ctx* ctx, int64_t nprob, int64_t n, int64_t r, bool aligned, bool overlap) {
  return aligned && !overlap && n % 8 == 0 && n >= 4096 && n <= (int64_t)kTrMaxCluster * kTrChunk && r > 0 && r < n &&
         nprob >= 2 * (int64_t)ctx->sm_count;
}
// does [p, p + bytes) overlap [o, o + bytes)
static bool spans_overlap(const void* p, const void* o, size_t bytes) {
  return p != nullptr && o != nullptr && (const char*)p < (const char*)o + bytes && (const char*)o < (const char*)p + bytes;
}

template <class R>
static int32_t prox_indballl0(spx_ctx* ctx, int64_t nprob, int64_t n, R* y, const R* xk, const R* sj, const R* q,
                              int64_t r, int32_t binf, double delta) {
  SPX_REQUIRE(ctx != nullptr, "null context");
  SPX_REQUIRE(nprob >= 0 && n >= 0, "negative size");
  if (nprob == 0 || n == 0) return SPX_OK;
  SPX_REQUIRE(y && xk && sj && q, "null device vector");
  DeviceGuard g(ctx->device);
  if (n > (int64_t)kTrMaxCluster * kTrChunk) {
    for (int64_t p = 0; p < nprob; ++p) {
      int32_t st = topr_global<R>(ctx, n, y + p * n, xk + p * n, sj + p * n, q + p * n, r, binf != 0, (R)delta);
      if (st != SPX_OK) return st;
    }
    return SPX_OK;
  }
  const uintptr_t bits = (uintptr_t)y | (uintptr_t)xk | (uintptr_t)sj | (uintptr_t)q;
  const bool vec = (bits & 15u) == 0 && (n * (int64_t)sizeof(R)) % 16 == 0;
  // batches: the stream form (one CTA per problem, several CTAs per SM)
  {
    const size_t bytes = (size_t)nprob * n * sizeof(R);
    const bool alias = spans_overlap(y, xk, bytes) || spans_overlap(y, sj, bytes) || spans_overlap(y, q, bytes);
    if (topr_stream_ok<R>(ctx, nprob, n, r, vec, alias)) {
      return binf ? topr_stream_launch<R, true>(ctx, nprob, n, y, xk, sj, q, r, (R)delta)
                  : topr_stream_launch<R, false>(ctx, nprob, n, y, xk, sj, q, r, (R)delta);
    }
  }
  if (binf) {
    return vec ? topr_cluster_launch<R, true, true>(ctx, nprob, n, y, xk, sj, q, r, (R)delta)
               : topr_cluster_launch<R, true, false>(ctx, nprob, n, y, xk, sj, q, r, (R)delta);
  }
  return vec ? topr_cluster_launch<R, false, true>(ctx, nprob, n, y, xk, sj, q, r, (R)delta)
             : topr_cluster_launch<R, false, false>(ctx, nprob, n, y, xk, sj, q, r, (R)delta);
}

// ψ(y) of the two types over the whole batch, as their ψ(y) entries compute it (the composed step's value)
static int32_t value_indballl0(spx_ctx* ctx, int64_t N, const double* xk, const double* sj, const double* y,
                               int32_t binf, double delta, int64_t r, double* out) {
  return binf ? spx_value_binf_f64(ctx, SPX_H_INDBALLL0, N, xk, sj, y, delta, r, 0, nullptr, nullptr, out)
              : spx_value_sep_f64(ctx, SPX_H_INDBALLL0, N, xk, sj, y, 0.0, r, out);
}
static int32_t value_indballl0(spx_ctx* ctx, int64_t N, const float* xk, const float* sj, const float* y, int32_t binf,
                               double delta, int64_t r, double* out) {
  return binf ? spx_value_binf_f32(ctx, SPX_H_INDBALLL0, N, xk, sj, y, delta, r, 0, nullptr, nullptr, out)
              : spx_value_sep_f32(ctx, SPX_H_INDBALLL0, N, xk, sj, y, 0.0, r, out);
}

// ---- the solver step of ShiftedIndBallL0 / ShiftedIndBallL0BInf (SURVEY.md 8f rank 1) -------------------------------
//     q = (-ν) ∇f;  prox!(s, ψ, q, ν);  xsy = (xk + sj) + s;  ψ(s);  Σ s²;  Σ ∇f·s
// A batch the stream form takes (topr_stream_ok, with xsy given and no output overlapping an input) runs it in ONE pass
// of the STEP form of topr_stream_kernel, then the radix kernel on the problems it flagged (in place: y = q = s) and
// topr_step_fixup_kernel for their xsy and sums: a fixed launch sequence, no host synchronisation until the fold.
// Every other call takes the composed form: spx_step_pre, prox! in place, the type's ψ(y), spx_step_post.
template <class R>
static int32_t step_indballl0(spx_ctx* ctx, int64_t nprob, int64_t n, R* s, R* xsy, const R* xk, const R* sj,
                              const R* grad, int64_t r, int32_t binf, double delta, double nu, double* out3) {
  SPX_REQUIRE(ctx != nullptr, "null context");
  SPX_REQUIRE(nprob >= 0 && n >= 0, "negative size");
  SPX_REQUIRE(out3 != nullptr, "null result array");
  const int64_t N = nprob * n;
  SPX_REQUIRE(N == 0 || (s && xk && sj && grad), "null device vector");
  const size_t bytes = (size_t)N * sizeof(R);
  SPX_REQUIRE(!spans_overlap(s, grad, bytes), "s must not alias grad");
  DeviceGuard g(ctx->device);
  out3[0] = out3[1] = out3[2] = 0.0;
  if (N == 0) return SPX_OK;
  const bool aligned = (((uintptr_t)s | (uintptr_t)xsy | (uintptr_t)xk | (uintptr_t)sj | (uintptr_t)grad) & 15u) == 0;
  const bool overlap = spans_overlap(s, xk, bytes) || spans_overlap(s, sj, bytes) || spans_overlap(xsy, xk, bytes) ||
                       spans_overlap(xsy, sj, bytes) || spans_overlap(xsy, grad, bytes) || spans_overlap(xsy, s, bytes);
  if (xsy != nullptr && topr_stream_ok<R>(ctx, nprob, n, r, aligned, overlap)) {
    TsStep<R> step{xsy, -(R)nu, 1.1 * (double)(R)delta, ctx->d_partials, 0};
    int grid = 0;
    const int32_t st = binf ? topr_stream_launch<R, true, true>(ctx, nprob, n, s, xk, sj, grad, r, (R)delta, step, &grid)
                            : topr_stream_launch<R, false, true>(ctx, nprob, n, s, xk, sj, grad, r, (R)delta, step, &grid);
    if (st != SPX_OK) return st;
    const int32_t st2 = finalize_partials(ctx, grid + ctx->sm_count, 2, false);
    if (st2 != SPX_OK) return st2;
    // the same predicates and scaling as ψ(y): ValueSep / scale_value, ValueBinfCount and its flag
    const double count = ctx->h_result[0].s;
    out3[0] = (binf && ctx->h_result[0].bad > 0) ? kInf : scale_value<R>(SPX_H_INDBALLL0, R(0), count, r);
    out3[1] = ctx->h_result[0].s2;
    out3[2] = ctx->h_result[1].s;
    return SPX_OK;
  }
  int32_t st = step_pre<R>(ctx, N, s, grad, nu);
  if (st != SPX_OK) return st;
  st = prox_indballl0<R>(ctx, nprob, n, s, xk, sj, s, r, binf, delta);
  if (st != SPX_OK) return st;
  st = value_indballl0(ctx, N, xk, sj, s, binf, delta, r, &out3[0]);
  if (st != SPX_OK) return st;
  double out2[2] = {0.0, 0.0};
  st = step_post<R>(ctx, N, xsy, xk, sj, s, grad, out2);
  if (st != SPX_OK) return st;
  out3[1] = out2[0];
  out3[2] = out2[1];
  return SPX_OK;
}

}  // namespace spx

using namespace spx;

#ifdef SPX_TR_TIMING
extern "C" int32_t spx_debug_topr_timing(unsigned long long* out8, int reset) {
  cudaMemcpyFromSymbol(out8, g_tr_t, 128);
  if (reset) {
    unsigned long long z[16] = {0};
    cudaMemcpyToSymbol(g_tr_t, z, 128);
  }
  return 0;
}
#endif
// Device self-test of the digit pick of the global path on a caller-supplied first-digit histogram (counts may
// exceed 2^31): returns the bin holding the `need`-th largest element and the number of elements above that bin.
extern "C" int32_t spx_selftest_topr_pick(spx_ctx* ctx, const uint64_t* hist_host, int64_t need, int32_t* bin_out,
                                          int64_t* above_out) {
  SPX_REQUIRE(ctx && hist_host && bin_out && above_out, "null argument");
  DeviceGuard g(ctx->device);
  int32_t st0 = ensure_scratch(ctx, sizeof(GlobalSel) + 4096);
  if (st0 != SPX_OK) return st0;
  GlobalSel* st = (GlobalSel*)ctx->d_scratch;
  static GlobalSel init;
  memset(&init, 0, sizeof(init));
  for (int b = 0; b < kTrBins; ++b) init.hist[b] = hist_host[b];
  init.need = need;
  init.shift = KeyTraits<double>::BITS;
  SPX_CUDA(cudaMemcpyAsync(st, &init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
  topr_g_pick<double><<<1, kPickThreads, 0, ctx->stream>>>(0, st);
  ctx->launches++;
  SPX_CUDA(cudaGetLastError());
  SPX_CUDA(cudaMemcpyAsync(&init, st, sizeof(init), cudaMemcpyDeviceToHost, ctx->stream));
  SPX_CUDA(cudaStreamSynchronize(ctx->stream));
  *bin_out = (int32_t)init.prefix;
  *above_out = need - init.need;
  return SPX_OK;
}
extern "C" int32_t spx_prox_indballl0_f64(spx_ctx* ctx, int64_t nprob, int64_t n, double* y, const double* xk,
                                          const double* sj, const double* q, int64_t r, int32_t binf, double delta) {
  return prox_indballl0<double>(ctx, nprob, n, y, xk, sj, q, r, binf, delta);
}
extern "C" int32_t spx_prox_indballl0_sharded_f64(spx_ctx* ctx, int64_t n_local, int64_t n_global, double* y,
                                                  const double* xk, const double* sj, const double* q, int64_t r,
                                                  int32_t binf, double delta, int32_t rank, int32_t world,
                                                  spx_allreduce_sum_fn reduce, void* user) {
  SPX_REQUIRE(ctx != nullptr, "null context");
  SPX_REQUIRE(n_local >= 0 && n_global >= n_local && world >= 1 && rank >= 0 && rank < world, "bad shard description");
  SPX_REQUIRE(n_local == 0 || (y && xk && sj && q), "null device vector");
  SPX_REQUIRE(world == 1 || reduce != nullptr || (ctx->comm != nullptr && ctx->comm_nranks == world),
              "a sharded vector needs the all-reduce callback or a communicator (spx_comm_init) of `world` ranks");
  DeviceGuard g(ctx->device);
  return topr_global<double>(ctx, n_local, y, xk, sj, q, r, binf != 0, delta, n_global, rank, world, reduce, user);
}
extern "C" int32_t spx_prox_indballl0_sharded_f32(spx_ctx* ctx, int64_t n_local, int64_t n_global, float* y,
                                                  const float* xk, const float* sj, const float* q, int64_t r,
                                                  int32_t binf, double delta, int32_t rank, int32_t world,
                                                  spx_allreduce_sum_fn reduce, void* user) {
  SPX_REQUIRE(ctx != nullptr, "null context");
  SPX_REQUIRE(n_local >= 0 && n_global >= n_local && world >= 1 && rank >= 0 && rank < world, "bad shard description");
  SPX_REQUIRE(n_local == 0 || (y && xk && sj && q), "null device vector");
  SPX_REQUIRE(world == 1 || reduce != nullptr || (ctx->comm != nullptr && ctx->comm_nranks == world),
              "a sharded vector needs the all-reduce callback or a communicator (spx_comm_init) of `world` ranks");
  DeviceGuard g(ctx->device);
  return topr_global<float>(ctx, n_local, y, xk, sj, q, r, binf != 0, (float)delta, n_global, rank, world, reduce,
                            user);
}
extern "C" int32_t spx_prox_indballl0_f32(spx_ctx* ctx, int64_t nprob, int64_t n, float* y, const float* xk,
                                          const float* sj, const float* q, int64_t r, int32_t binf, double delta) {
  return prox_indballl0<float>(ctx, nprob, n, y, xk, sj, q, r, binf, delta);
}
extern "C" int32_t spx_step_indballl0_f64(spx_ctx* ctx, int64_t nprob, int64_t n, double* s, double* xsy,
                                          const double* xk, const double* sj, const double* grad, int64_t r,
                                          int32_t binf, double delta, double nu, double* out3) {
  return step_indballl0<double>(ctx, nprob, n, s, xsy, xk, sj, grad, r, binf, delta, nu, out3);
}
extern "C" int32_t spx_step_indballl0_f32(spx_ctx* ctx, int64_t nprob, int64_t n, float* s, float* xsy,
                                          const float* xk, const float* sj, const float* grad, int64_t r,
                                          int32_t binf, double delta, double nu, double* out3) {
  return step_indballl0<float>(ctx, nprob, n, s, xsy, xk, sj, grad, r, binf, delta, nu, out3);
}
