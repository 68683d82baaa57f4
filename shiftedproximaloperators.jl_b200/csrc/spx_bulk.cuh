// spx_bulk.cuh -- the bulk-copy ring form of the elementwise streaming kernel (ew_bulk_kernel).
//
// In ew_kernel a warp issues its loads, waits, then computes with nothing in flight, and the registers of the Box
// functors (64-80) cap how many warps can wait at once, so HBM idles part of each tile.  Here the loads are taken off
// the compute warps: one producer warp per CTA keeps a ring of ST stages full with cp.async.bulk copies (one elected
// lane, NIN contiguous runs of TILE bytes per stage, all completing on the stage's `full` mbarrier), and CW consumer
// warps read the stage
// with 16-byte shared loads, call the same functor on the same global index as ew_kernel (so every output is
// bit-identical), write y with streaming stores and release the stage on its `empty` mbarrier.  Bytes in flight per
// SM are CTAS x ST x NIN x TILE whatever the functor's register count.
// Schedule: tile t (TILE / sizeof(R) elements of every operand) belongs to CTA t % gridDim.x; the producer and every
// consumer run the same loop over the CTA's tiles, so trip counts and barrier phases agree by construction, and the
// ψ partials keep one slot per CTA in a fixed order.  The n % TE elements past the last full tile are taken by the
// last CTA's consumers with plain loads.  Every operand must be a 16-byte-aligned vector (ew_launch checks).
// Operators opt in with `static constexpr bool BULK = true`.  It pays where the functor is light enough for 16 warps
// per SM (L0Box/L1Box prox!, L0Box iprox!); issue-bound functors (RootNormLhalfBox) keep ew_kernel's 32 warps.
// The SPX_EWB_* sizes are A/B-able with `tools/build_variant.sh NAME "-DSPX_EWB_...=..." spx_bulk.cu`.
#pragma once
#include "spx_common.cuh"

namespace spx {

#ifndef SPX_EWB_TILE
#define SPX_EWB_TILE 8192  // bytes of one operand per stage (1024 Float64 / 2048 Float32 elements)
#endif
#ifndef SPX_EWB_STAGES
#define SPX_EWB_STAGES 3
#endif
#ifndef SPX_EWB_WARPS
#define SPX_EWB_WARPS 16  // consumer warps per CTA (+ one producer warp)
#endif
#ifndef SPX_EWB_CTAS
#define SPX_EWB_CTAS 1  // resident CTAs per SM (also the __launch_bounds__ min-blocks)
#endif

template <class Op, int TILE = SPX_EWB_TILE, int ST = SPX_EWB_STAGES, int CW = SPX_EWB_WARPS, int CTAS = SPX_EWB_CTAS>
__global__ void __launch_bounds__((CW + 1) * 32, CTAS)
    ew_bulk_kernel(const Op op, const long long n, const long long index_base, Partial* __restrict__ partials) {
  using R = typename Op::Real;
  constexpr int NIN = Op::NIN, VEC = 16 / (int)sizeof(R);
  constexpr int TE = TILE / (int)sizeof(R);  // elements of one operand per tile
  constexpr int PK = TILE / 16;              // 16-byte packets of one operand per tile
  constexpr int NCT = CW * 32;               // consumer threads
  static_assert(TILE % 16 == 0 && ST >= 2, "bulk copies move 16-byte granules");
  extern __shared__ __align__(128) unsigned char ewb_smem[];  // ST x NIN x TILE
  __shared__ __align__(8) uint64_t full[ST], empty[ST];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < ST; ++s) {
      mbar_init(&full[s], 1);    // the producer's arrive.expect_tx; the copies' bytes complete the phase
      mbar_init(&empty[s], CW);  // one arrive per consumer warp
    }
  }
  __syncthreads();
  Partial acc;
  acc.s = 0.0;
  acc.s2 = 0.0;
  acc.bad = -1;
  const long long ntiles = n / TE;
  if (warp == CW) {
    if (lane == 0) {
      int s = 0;
      uint32_t round = 0;  // completed passes over the ring
      for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
        if (round > 0) mbar_wait(&empty[s], (round - 1) & 1u);  // the consumers' release of pass round - 1
        fence_proxy_async();
        mbar_expect_tx(&full[s], (uint32_t)(NIN * TILE));
        unsigned char* const buf = ewb_smem + (size_t)s * NIN * TILE;
#pragma unroll
        for (int k = 0; k < NIN; ++k) bulk_g2s(buf + k * TILE, op.in[k] + t * TE, (uint32_t)TILE, &full[s]);
        if (++s == ST) {
          s = 0;
          ++round;
        }
      }
    }
  } else {
    const int ct = threadIdx.x;  // consumer thread 0 .. NCT-1
    const uint32_t smem0 = smem_u32(ewb_smem);
    int s = 0;
    uint32_t round = 0;
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
      mbar_wait(&full[s], round & 1u);
      const uint32_t buf = smem0 + (uint32_t)(s * NIN * TILE);
      for (int p = ct; p < PK; p += NCT) {
        Pack<R, VEC> reg[NIN];
#pragma unroll
        for (int k = 0; k < NIN; ++k) lds16(buf + (uint32_t)(k * TILE + p * 16), reg[k]);
        const long long v = t * PK + p;  // packet index in the operand
        Pack<R, VEC> out;
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
          R x[NIN];
#pragma unroll
          for (int k = 0; k < NIN; ++k) x[k] = reg[k].v[e];
          out.v[e] = op.apply(x, index_base + v * VEC + e, acc);
        }
        if (Op::OUT) st_stream(op.y + v * VEC, out);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[s]);
      if (++s == ST) {
        s = 0;
        ++round;
      }
    }
    // the partial tile: the last CTA's consumers, plain loads
    if (blockIdx.x == gridDim.x - 1) {
      for (long long i = ntiles * TE + ct; i < n; i += NCT) {
        R x[NIN];
#pragma unroll
        for (int k = 0; k < NIN; ++k) x[k] = op.in[k][i];
        R o = op.apply(x, index_base + i, acc);
        if (Op::OUT) op.y[i] = o;
      }
    }
  }
  if (Op::ACC) {
    acc = block_fold<(CW + 1) * 32>(acc);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc;
  }
}

// dynamic shared memory of one CTA: ST stages of NIN operand runs of TILE bytes
template <class Op, int TILE = SPX_EWB_TILE, int ST = SPX_EWB_STAGES> constexpr size_t ew_bulk_smem() {
  return (size_t)ST * Op::NIN * TILE;
}

// Launch `op` over n >= one tile of elements (ew_launch's routing).  The dynamic shared memory attribute is set on
// every launch: it belongs to the current device, and one process may drive several.  Grid = SPX_EWB_CTAS per SM, at
// most one CTA per tile; the static schedule needs no co-residency, so a grid larger than what fits is still correct.
template <class Op>
int32_t ew_bulk_launch(spx_ctx* ctx, cudaStream_t stream, const Op& op, int64_t n, int64_t index_base, Partial* partials,
                       int* nblocks_out) {
  using R = typename Op::Real;
  constexpr size_t smem = ew_bulk_smem<Op>();
  static_assert(smem <= 227 * 1024, "ring larger than the shared memory of one CTA");
  auto kern = ew_bulk_kernel<Op>;
  if (nblocks_out) *nblocks_out = 0;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "ew_bulk_kernel shared memory attribute");
  const long long ntiles = n / (SPX_EWB_TILE / (int)sizeof(R));
  long long cap = (long long)ctx->sm_count * SPX_EWB_CTAS;
  if (cap > kMaxPartials) cap = kMaxPartials;
  const int grid = (int)(ntiles < 1 ? 1 : (ntiles < cap ? ntiles : cap));
  kern<<<grid, (SPX_EWB_WARPS + 1) * 32, smem, stream>>>(op, n, index_base, partials);
  ctx->launches++;
  if (nblocks_out) *nblocks_out = grid;
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "ew_bulk_kernel launch");
  return SPX_OK;
}

}  // namespace spx
