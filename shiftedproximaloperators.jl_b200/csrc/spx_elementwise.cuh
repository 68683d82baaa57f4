// spx_elementwise.cuh -- the one streaming kernel every separable operator runs on.
//
// Each operand is a contiguous stream read exactly once with 128-bit loads
// (2 x f64 / 4 x f32 per thread per request, UNROLL independent requests per
// stream in flight before the first use), the result is written once with a
// 128-bit streaming store, and the optional ψ(y) partial sum is folded in the
// same pass (warp shuffle -> block -> one slot per block, fixed order).
// Grid = resident CTAs per SM x 148 SMs, grid-stride over tiles.
#pragma once
#include <type_traits>

#include "spx_common.cuh"

namespace spx {

constexpr int kEwThreads = 256;

// Op concept:
//   using Real = R;  static constexpr int NIN; static constexpr bool OUT, ACC;
//   const R* in[NIN]; R fill[NIN]; R* y;
//   __device__ R apply(const R (&x)[NIN], long long i, Partial& acc) const;
// resident CTAs per SM an operator asks for (Op::MINB, default 1 = let ptxas choose registers)
template <class Op, class = void> struct MinBlocks { static constexpr int value = 1; };
template <class Op> struct MinBlocks<Op, std::void_t<decltype(Op::MINB)>> { static constexpr int value = Op::MINB; };

// NPTR: number of leading operands known to be vectors, the others being scalars (fill) -- resolved at
// compile time so the streaming loop carries no null tests, no fill moves and no predicated address
// arithmetic (~10 % of the instructions of a Box kernel); NPTR < 0 keeps the run-time tests.
template <class Op, class = void> struct SplitNull { static constexpr bool value = false; };
template <class Op> struct SplitNull<Op, std::void_t<decltype(Op::SPLIT_NULL)>> { static constexpr bool value = Op::SPLIT_NULL; };

// Operators that declare `static constexpr bool PACKET = true` (and `int PREFETCH, L2_AHEAD`) are applied one 128-bit
// packet at a time in the vector launches, in four parts (see ProxLhalfBox):
//   bool selects_all()                       every element selected: the loop then holds no selection test at all
//   bool pick_packet(x, o, hard)             the common path: o for every element, true if some element needs the slow path
//   void exact_packet(x, o, hard)            the slow path, only when pick_packet returned true
//   Pack finish_packet<ALL>(x, o, i0, acc)   the selection and the ψ terms
// After the slow path the packet is loaded again rather than held across it: held, it pushes the common path's registers
// to the stack.  With PREFETCH = 1 each thread also issues the loads of its next packet before it computes the
// current one (NIN x 16 bytes more in registers).  With L2_AHEAD = k > 0 it asks L2 for the lines of its packet k
// iterations ahead (`prefetch.global.L2`: no register, no shared memory), so its own loads later hit L2.
template <class Op, class = void> struct Packet { static constexpr bool value = false; };
template <class Op> struct Packet<Op, std::void_t<decltype(Op::PACKET)>> { static constexpr bool value = Op::PACKET; };

template <int VEC, int NPTR, class Op>
__device__ __forceinline__ void ew_load_packet(const Op& op, long long v, long long nvec,
                                               Pack<typename Op::Real, VEC> (&x)[Op::NIN]) {
#pragma unroll
  for (int k = 0; k < Op::NIN; ++k) {
    if (NPTR >= 0) {
      if (k < NPTR) {
        if (v < nvec) ld_stream(op.in[k] + v * VEC, x[k]);  // past the end: never used
      } else {
#pragma unroll
        for (int e = 0; e < VEC; ++e) x[k].v[e] = op.fill[k];
      }
    } else if (op.in[k] != nullptr && v < nvec) {
      ld_stream(op.in[k] + v * VEC, x[k]);
    } else {
#pragma unroll
      for (int e = 0; e < VEC; ++e) x[k].v[e] = op.fill[k];
    }
  }
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

template <int VEC, int NPTR, bool ALL, class Op>
__device__ __forceinline__ void ew_packet_loop(const Op& op, long long nvec, long long index_base, Partial& acc) {
  using R = typename Op::Real;
  const long long stride = (long long)gridDim.x * kEwThreads;
  long long v = (long long)blockIdx.x * kEwThreads + threadIdx.x;
  Pack<R, VEC> x[Op::NIN];
  if (Op::PREFETCH > 0) ew_load_packet<VEC, NPTR>(op, v, nvec, x);
  for (; v < nvec; v += stride) {
    if (Op::L2_AHEAD > 0) {
      const long long va = v + Op::L2_AHEAD * stride;
      if (va < nvec) {
#pragma unroll
        for (int k = 0; k < Op::NIN; ++k)
          if (NPTR >= 0 ? k < NPTR : op.in[k] != nullptr) prefetch_l2(op.in[k] + va * VEC);
      }
    }
    Pack<R, VEC> nx[Op::NIN];
    if (Op::PREFETCH > 0)
      ew_load_packet<VEC, NPTR>(op, v + stride, nvec, nx);
    else
      ew_load_packet<VEC, NPTR>(op, v, nvec, x);
    Pack<R, VEC> o;
    bool hard[VEC];
    if (op.pick_packet(x, o, hard)) {
      op.exact_packet(x, o, hard);
      // the same bytes: this thread stores packet v below and packet v + stride in its next iteration (y may alias q)
      ew_load_packet<VEC, NPTR>(op, v, nvec, x);
      if (Op::PREFETCH > 0) ew_load_packet<VEC, NPTR>(op, v + stride, nvec, nx);
    }
    const Pack<R, VEC> out = op.template finish_packet<ALL>(x, o, index_base + v * VEC, acc);
    if (Op::OUT) st_stream(op.y + v * VEC, out);
    if (Op::PREFETCH > 0) {
#pragma unroll
      for (int k = 0; k < Op::NIN; ++k) x[k] = nx[k];
    }
  }
}

template <int VEC, int UNROLL, class Op, int NPTR = -1>
__global__ void __launch_bounds__(kEwThreads, MinBlocks<Op>::value)
    ew_kernel(const Op op, const long long n, const long long index_base, Partial* __restrict__ partials) {
  using R = typename Op::Real;
  constexpr int NIN = Op::NIN;
  Partial acc;
  acc.s = 0.0;
  acc.s2 = 0.0;
  acc.bad = -1;

  const long long nvec = n / VEC;
  const long long tile = (long long)kEwThreads * UNROLL;
  if constexpr (Packet<Op>::value && VEC > 1) {
    static_assert(UNROLL == 1, "the packet loop strides by one packet per thread");
    if (op.selects_all())
      ew_packet_loop<VEC, NPTR, true>(op, nvec, index_base, acc);
    else
      ew_packet_loop<VEC, NPTR, false>(op, nvec, index_base, acc);
  } else {
    for (long long base = (long long)blockIdx.x * tile; base < nvec; base += (long long)gridDim.x * tile) {
      Pack<R, VEC> reg[NIN][UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        const long long v = base + (long long)u * kEwThreads + threadIdx.x;
#pragma unroll
        for (int k = 0; k < NIN; ++k) {
          if (NPTR >= 0) {  // vector-ness known at compile time: no fill moves, no null tests
            if (k < NPTR) {
              if (v < nvec) ld_stream(op.in[k] + v * VEC, reg[k][u]);  // past the end: never used below
            } else {
#pragma unroll
              for (int e = 0; e < VEC; ++e) reg[k][u].v[e] = op.fill[k];
            }
          } else if (op.in[k] != nullptr && v < nvec) {  // one predicate: keeps every load of the tile in one batch
            ld_stream(op.in[k] + v * VEC, reg[k][u]);
          } else {
#pragma unroll
            for (int e = 0; e < VEC; ++e) reg[k][u].v[e] = op.fill[k];
          }
        }
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        const long long v = base + (long long)u * kEwThreads + threadIdx.x;
        if (v < nvec) {
          Pack<R, VEC> out;
#pragma unroll
          for (int e = 0; e < VEC; ++e) {
            R x[NIN];
#pragma unroll
            for (int k = 0; k < NIN; ++k) x[k] = reg[k][u].v[e];
            out.v[e] = op.apply(x, index_base + v * VEC + e, acc);
          }
          if (Op::OUT) st_stream(op.y + v * VEC, out);
        }
      }
    }
  }
  // scalar tail (n not a multiple of VEC): the last block's first threads
  if (VEC > 1 && blockIdx.x == gridDim.x - 1) {
    const long long i = nvec * VEC + threadIdx.x;
    if (i < n) {
      R x[NIN];
#pragma unroll
      for (int k = 0; k < NIN; ++k) x[k] = op.in[k] != nullptr ? op.in[k][i] : op.fill[k];
      R o = op.apply(x, index_base + i, acc);
      if (Op::OUT) op.y[i] = o;
    }
  }
  if (Op::ACC) {
    acc = block_fold<kEwThreads>(acc);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc;
  }
}

// ------------------------------------------------------------------ bulk-copy ring --
// Operators that declare `static constexpr bool BULK = true` stream their operands through ew_bulk_kernel (spx_bulk.cuh)
// when every operand is a 16-byte-aligned vector and n >= SPX_EWB_MIN_N.  The kernel and its launches live in their own
// translation unit, spx_bulk.cu, which instantiates ew_bulk_launch for those operators: its dynamic shared memory
// (`extern __shared__`) makes nvcc reserve 1 KiB of static shared memory in every kernel of the module it is in.
#ifndef SPX_EWB_MIN_N
#define SPX_EWB_MIN_N (1 << 20)  // elements: where the ring starts to beat ew_kernel (profiles/README.md, round 3)
#endif
template <class Op, class = void> struct Bulk { static constexpr bool value = false; };
template <class Op> struct Bulk<Op, std::void_t<decltype(Op::BULK)>> { static constexpr bool value = Op::BULK; };
template <class Op>
int32_t ew_bulk_launch(spx_ctx* ctx, cudaStream_t stream, const Op& op, int64_t n, int64_t index_base, Partial* partials,
                       int* nblocks_out);

template <class Op> inline bool aligned16(const Op& op) {
  uintptr_t bits = 0;
  for (int k = 0; k < Op::NIN; ++k) bits |= (uintptr_t)op.in[k];
  if (Op::OUT) bits |= (uintptr_t)op.y;
  return (bits & 15u) == 0;
}

template <int VEC, int UNROLL, class Op, int NPTR = -1> inline int ew_blocks_per_sm() {
  static int cached = 0;  // per instantiation
  if (cached == 0) {
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, ew_kernel<VEC, UNROLL, Op, NPTR>, kEwThreads, 0) !=
            cudaSuccess ||
        nb < 1)
      nb = 1;
    cached = nb;
  }
  return cached;
}

// how many leading operands are vectors, or -1 if a scalar operand precedes a vector
template <class Op> inline int leading_vectors(const Op& op) {
  int k = 0;
  while (k < Op::NIN && op.in[k] != nullptr) ++k;
  for (int j = k; j < Op::NIN; ++j)
    if (op.in[j] != nullptr) return -1;
  return k;
}

// Launch `op` over n elements on `stream`.  Returns the number of blocks (=
// number of partial slots written when Op::ACC) through nblocks_out.
template <class Op>
int32_t ew_launch(spx_ctx* ctx, cudaStream_t stream, const Op& op, int64_t n, int64_t index_base,
                  Partial* partials, int* nblocks_out) {
  using R = typename Op::Real;
  constexpr int VECW = 16 / (int)sizeof(R);
  constexpr int UNROLL = Op::UNROLL;
  if (nblocks_out) *nblocks_out = 0;
  if (n <= 0) return SPX_OK;
  const bool vec = aligned16(op);
  if constexpr (Bulk<Op>::value) {
    if (vec && n >= SPX_EWB_MIN_N && leading_vectors(op) == Op::NIN)
      return ew_bulk_launch(ctx, stream, op, n, index_base, partials, nblocks_out);
  }
  const long long nvec = vec ? n / VECW : n;
  const long long tile = (long long)kEwThreads * UNROLL;
  long long want = (nvec + tile - 1) / tile;
  if (want < 1) want = 1;
  // operators with nullable trailing operands (the Box bounds): all vectors, or exactly the last two scalar
  int nptr = -1;
  if constexpr (SplitNull<Op>::value) {
    const int lead = leading_vectors(op);
    if (vec && (lead == Op::NIN || lead == Op::NIN - 2)) nptr = lead;
  }
  int per_sm = !vec ? ew_blocks_per_sm<1, UNROLL, Op>()
                    : (nptr < 0 ? ew_blocks_per_sm<VECW, UNROLL, Op>()
                                : (nptr == Op::NIN ? ew_blocks_per_sm<VECW, UNROLL, Op, Op::NIN>()
                                                   : ew_blocks_per_sm<VECW, UNROLL, Op, Op::NIN - 2>()));
  long long cap = (long long)ctx->sm_count * per_sm;
  if (cap > kMaxPartials) cap = kMaxPartials;
  int grid = (int)(want < cap ? want : cap);
  if (!vec)
    ew_kernel<1, UNROLL, Op><<<grid, kEwThreads, 0, stream>>>(op, n, index_base, partials);
  else if (nptr < 0)
    ew_kernel<VECW, UNROLL, Op><<<grid, kEwThreads, 0, stream>>>(op, n, index_base, partials);
  else if (nptr == Op::NIN)
    ew_kernel<VECW, UNROLL, Op, Op::NIN><<<grid, kEwThreads, 0, stream>>>(op, n, index_base, partials);
  else
    ew_kernel<VECW, UNROLL, Op, Op::NIN - 2><<<grid, kEwThreads, 0, stream>>>(op, n, index_base, partials);
  ctx->launches++;
  if (nblocks_out) *nblocks_out = grid;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "ew_kernel launch");
  return SPX_OK;
}

}  // namespace spx
