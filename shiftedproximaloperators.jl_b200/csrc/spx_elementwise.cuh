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
