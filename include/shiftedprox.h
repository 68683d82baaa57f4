/* ============================================================================
 * shiftedprox.h -- C ABI of libshiftedprox.so (hand-written sm_100a CUDA).
 *
 * Drop-in boundary for the shifted prox hot path of ShiftedProximalOperators.jl
 * v0.2.2.  The reference is pure Julia with no FFI on this path; the entry
 * points below are what a Julia glue package binds with
 *   ccall((:spx_..., libshiftedprox), Int32, (...), ...)
 * in place of the method bodies cited at each declaration (file:line relative
 * to the reference tree).  The in-tree FFI precedent the style follows is
 * src/psvd.jl:99-137 (status out of the callee + a `chk...error` on the Julia
 * side).  INTEGRATION.md shows the binding.
 *
 * Conventions
 *  - every function returns int32 status: 0 = ok, <0 = SPX_E_* below,
 *    >0 = a cudaError_t; spx_last_error() returns a thread-local message.
 *  - `R*` arguments are DEVICE pointers on the context's device unless the
 *    name ends in `_host`.  The library never frees or retains caller
 *    pointers beyond a call.
 *  - calls are enqueued on the context's stream and are asynchronous unless
 *    they return a scalar to the host (`psi_out`, `*_out`), in which case
 *    they synchronise that stream before returning.
 *  - scalars (lambda, sigma, delta, bounds) are passed as double and rounded
 *    to the element type R inside (the reference constrains them to R).
 *  - indices are 0-based; `n` is the vector length.
 *  - arithmetic follows the reference operation by operation (no FMA
 *    contraction, Julia min/max/sign semantics); see DESIGN.md.
 *  - a ψ must not be used from two host threads at once (the reference is
 *    not re-entrant per ψ either: scratch lives in the struct).
 * ========================================================================== */
#ifndef SHIFTEDPROX_H
#define SHIFTEDPROX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPX_OK 0
#define SPX_E_INVALID (-1)    /* bad argument (null pointer, n < 0, unknown kind ...) */
#define SPX_E_ASSERT_D (-2)   /* `@assert d[i] > 0` failed: shiftedNormL1.jl:70, shiftedNormL0.jl:70 */
#define SPX_E_BOUNDS (-3)     /* some l[i] > u[i]: shiftedNormL0Box.jl:33-35, shiftedNormL1Box.jl:33-35 */
#define SPX_E_NOROOT (-4)     /* trust-region root finder did not bracket a root */
#define SPX_E_UNSUPPORTED (-5)

typedef struct spx_ctx spx_ctx; /* one device, one stream, reduction scratch */

/* `l` / `u` of the Box types are "scalar or vector" (untyped struct parameters
 * V3, V4: shiftedNormL1Box.jl:3-19).  vec == NULL -> the scalar `val`. */
typedef struct spx_bound {
  const void* vec; /* device pointer to n elements of R, or NULL */
  double val;
} spx_bound;

/* `selected::AbstractArray{<:Integer}` (shiftedNormL1Box.jl:10,19,106,71).
 *  SPX_SEL_ALL   every index (the default `1:length(xk)`)
 *  SPX_SEL_RANGE start:step:stop, 0-based inclusive (e.g. Julia `1:2:n` -> 0,2,n-1)
 *  SPX_SEL_MASK  bit i of mask[i/32] set <=> i selected (built by spx_build_mask from
 *                any index list; membership is what prox!/iprox! need, :106)
 *  For ψ(y) of a list with duplicates (the gather `x[selected]` counts them
 *  twice, :71) pass the list as well: `list`/`nlist` (device, int64, 0-based). */
#define SPX_SEL_ALL 0
#define SPX_SEL_RANGE 1
#define SPX_SEL_MASK 2
typedef struct spx_sel {
  int32_t kind;
  int64_t start, step, stop;
  const uint32_t* mask; /* device, ceil(n/32) words */
  const int64_t* list;  /* device, optional (values only) */
  int64_t nlist;
} spx_sel;

/* Sum all-reduce supplied by the host when one vector is sharded over several
 * GPUs (one process per GPU): must replace vals[0..count) by their sum over all
 * ranks, identically on every rank (e.g. ncclAllReduce / torch.distributed
 * all_reduce on a Float64 buffer).  Return 0 on success. */
typedef int32_t (*spx_allreduce_sum_fn)(void* user, double* vals, int32_t count);

/* h kinds for the value entry points */
#define SPX_H_L1 0        /* NormL1(λ):        λ‖v‖₁            (ProximalOperators 0.15) */
#define SPX_H_L0 1        /* NormL0(λ):        λ·count(v≠0)                              */
#define SPX_H_LHALF 2     /* RootNormLhalf(λ): λ Σ√|v|          (rootNormLhalf.jl:27-29) */
#define SPX_H_INDBALLL0 3 /* IndBallL0(r):     count(v≠0) ≤ r ? 0 : Inf                  */
#define SPX_H_GROUPL2 4   /* GroupNormL2:      Σ_g λ_g‖v_g‖₂    (groupNormL2.jl:33-39)   */

/* ------------------------------------------------------------- context --- */
int32_t spx_version(void);
const char* spx_last_error(void);
/* stream: the cudaStream_t to enqueue on, e.g. the host framework's current
 * stream; NULL is CUDA's default stream (stream 0), as everywhere in the CUDA
 * API.  own_stream != 0: ignore `stream`, the context creates (and later
 * destroys) its own non-blocking stream. */
int32_t spx_ctx_create(spx_ctx** out, int32_t device, void* stream, int32_t own_stream);
int32_t spx_ctx_destroy(spx_ctx* ctx);
int32_t spx_ctx_set_stream(spx_ctx* ctx, void* stream);
int32_t spx_ctx_synchronize(spx_ctx* ctx);
int32_t spx_ctx_sm_count(spx_ctx* ctx, int32_t* out);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int32_t spx_ctx_launch_count(spx_ctx* ctx, int64_t* out);

/* ------------------------------------------- multi-GPU (one process per GPU) ---
 * The reference is single-process; SURVEY.md §8e shards a vector (or a batch) contiguously over the GPUs of a box.
 * The path's only exchanges are scalars -- ψ(y) partial sums + infeasibility flag
 * (ShiftedProximalOperators.jl:51-54 and the Box / BInf overrides), the partial sums of every pass of the ℓ2
 * trust-region search (shiftedNormL1B2.jl:53-62), the fused step's three scalars -- and the digit histograms of a
 * single-vector top-r (shiftedIndBallL0.jl:66-70).  With a communicator attached to the context they are
 * all-reduced ON THE DEVICE (ncclAllReduce over NVLink on the context's stream, directly on the folded slots, sum
 * for Σ and max for the flag so `Inf` survives) before the one D2H copy of the call.  NCCL is bound at run time
 * (dlopen); rank 0 creates the id, the host passes its 128 bytes to the other ranks by any means. */
#define SPX_COMM_ID_BYTES 128
int32_t spx_comm_available(void);              /* 1 if libnccl.so.2 could be bound */
int32_t spx_comm_unique_id(void* id_out128);   /* ncclGetUniqueId */
int32_t spx_comm_init(spx_ctx* ctx, int32_t nranks, int32_t rank, const void* id128);
int32_t spx_comm_destroy(spx_ctx* ctx);
/* on != 0: every scalar a call hands back (psi_out, *_out of the value entry points, out3_host of the fused step,
 * the decisions of spx_prox_l1b2_*) is the value over ALL shards, identical on every rank; every rank must then
 * make the same calls in the same order.  on == 0: per-shard values (the default). */
int32_t spx_comm_reduce_scalars(spx_ctx* ctx, int32_t on);
int32_t spx_comm_info(spx_ctx* ctx, int32_t* nranks_out, int32_t* rank_out, int64_t* collectives_out);
/* Peer-memory exchange (optional, on top of or instead of the NCCL communicator): every rank exports the IPC handle of
 * its exchange buffer, the host passes the nranks handles around (rank order), every rank maps them.  The scalar
 * reductions (1..16 slots of {Σ, Σ₂, flag}) are then finished by the fold kernel itself: stores into every peer's
 * buffer over NVLink, a spin on the own buffer, the sum in rank order -- no separate collective launch. */
#define SPX_PEER_HANDLE_BYTES 64
int32_t spx_comm_peer_export(spx_ctx* ctx, void* handle_out64);
int32_t spx_comm_peer_attach(spx_ctx* ctx, int32_t nranks, int32_t rank, const void* handles /* nranks x 64 bytes */);
int32_t spx_comm_peer_detach(spx_ctx* ctx);
int32_t spx_comm_peer_active(spx_ctx* ctx); /* 1 when the scalar reductions go over the exchange buffers */
/* building block: in-place all-reduce of `count` doubles in device memory, enqueued on the context's stream
 * (op 0 = sum, 1 = max); a context without communicator leaves the buffer as is */
int32_t spx_comm_allreduce_f64(spx_ctx* ctx, double* dev_buf, int64_t count, int32_t op);

/* ----------------------------------------- device buffers (Julia owns) --- */
/* replaces `similar(xk)` / `zero(xk)` in the constructors, e.g. shiftedNormL1.jl:16-29 */
int32_t spx_malloc(spx_ctx* ctx, size_t bytes, void** out);
int32_t spx_free(spx_ctx* ctx, void* p);
int32_t spx_malloc_host(size_t bytes, void** out); /* pinned host memory */
int32_t spx_free_host(void* p);
int32_t spx_memcpy_h2d(spx_ctx* ctx, void* dst, const void* src_host, size_t bytes);
int32_t spx_memcpy_d2h(spx_ctx* ctx, void* dst_host, const void* src, size_t bytes); /* synchronises */
/* `shift!`: ψ.xk .= v / ψ.sj .= v   (ShiftedProximalOperators.jl:72-79) and
 * vector `set_bounds!` (ShiftedProximalOperators.jl:107-111) */
int32_t spx_memcpy_d2d(spx_ctx* ctx, void* dst, const void* src, size_t bytes);
/* dst[i * dst_stride] = src[i * src_stride], i < n (strides in elements of elem_bytes = 4 or 8 bytes): gather of a
 * strided `SubArray` shift (`x = view(y, 1:2:10); shifted(h, x)`, test/runtests.jl:199-200) into the contiguous
 * shadow the kernels read, and the scatter back after `shift!` writes it */
int32_t spx_copy_strided(spx_ctx* ctx, int64_t n, int32_t elem_bytes, void* dst, int64_t dst_stride,
                         const void* src, int64_t src_stride);
int32_t spx_fill_f64(spx_ctx* ctx, double* p, int64_t n, double v);
int32_t spx_fill_f32(spx_ctx* ctx, float* p, int64_t n, float v);
/* ctor validation `any(l .> u)` (shiftedNormL1Box.jl:33, shiftedNormL0Box.jl:33); *out = 1 if any */
int32_t spx_any_gt_f64(spx_ctx* ctx, int64_t n, const spx_bound* l, const spx_bound* u, int32_t* out);
int32_t spx_any_gt_f32(spx_ctx* ctx, int64_t n, const spx_bound* l, const spx_bound* u, int32_t* out);
/* membership bitmask of an arbitrary index list (device int64, 0-based, any
 * order, duplicates allowed); mask has ceil(n/32) words and is zeroed first */
int32_t spx_build_mask(spx_ctx* ctx, int64_t n, const int64_t* list, int64_t nlist, uint32_t* mask);
/* synthetic inputs of SURVEY.md §8d, bit-identical to the oracle's generator:
 * out[i] = scale * u(i0 + i, stream) + shift,  u = (splitmix64(...) >> 11) * 2^-53 */
int32_t spx_fill_uniform_f64(spx_ctx* ctx, double* out, int64_t n, int64_t i0, uint64_t seed,
                             uint64_t stream, double scale, double shift);
int32_t spx_fill_uniform_f32(spx_ctx* ctx, float* out, int64_t n, int64_t i0, uint64_t seed,
                             uint64_t stream, float scale, float shift);
/* Device self-test of the FP64 building blocks the kernels use instead of library calls: on n
 * pseudo-random operands, counts results that differ from the IEEE operation in any bit.
 * mismatches_out[0]: branch-free sqrt vs sqrt();  [1]: reciprocal + two Markstein corrections vs a/d;
 * [2]: uniform-divisor quotient vs a/s.  All three must be 0. */
int32_t spx_selftest_math(spx_ctx* ctx, int64_t n, uint64_t seed, int64_t* mismatches_out);
/* Device self-test of the digit pick of the single-vector top-r path (spx_prox_indballl0_* with one long vector and
 * its sharded form): hist_host holds 2048 counts, most significant digit first by bin index, possibly above 2^31;
 * returns the bin that holds the need-th largest element and the number of elements in the bins above it. */
int32_t spx_selftest_topr_pick(spx_ctx* ctx, const uint64_t* hist_host, int64_t need, int32_t* bin_out,
                               int64_t* above_out);
/* GroupNormL2's constructor checks (groupNormL2.jl:20-23) for the device layout: offs (device int64, ngroups + 1 entries)
 * must start at 0, never decrease and end at n; SPX_E_INVALID otherwise.  Call once when ψ is built: the prox!/ψ(y)
 * entry points trust the offsets.  The same pass records, per context, which group-size classes the layout holds
 * (keyed on offs / ngroups / n), so that later calls launch only the kernels that have work; a layout never
 * validated, or changed afterwards, is still computed correctly -- every class is launched, or the warp kernels take
 * over the groups of a class that was skipped.  Index sets that are not contiguous ranges in order (the reference accepts any
 * `idx`) cannot be expressed as CSR offsets: the host layer rejects them at construction. */
int32_t spx_group_validate_offsets(spx_ctx* ctx, int64_t n, int64_t ngroups, const int64_t* offs);
/* order-independent 64-bit checksum of a buffer's bits (Σ mix(word_i, i) mod 2^64),
 * identical to oracle.checksum(); used for full-size parity */
int32_t spx_checksum(spx_ctx* ctx, const void* p, int64_t nwords64, uint64_t* out);

/* ------------------------------------------------ separable prox (a2-a6) ---
 * psi_out (host, may be NULL): if given, ψ(y) at the freshly computed y is
 * accumulated in the same pass (ShiftedProximalOperators.jl:51-54 fused) and
 * the call synchronises. */
/* one operation of spx_box_multi_host_*: op 0 L1Box, 1 L0Box, 2 LhalfBox; d_host == NULL -> */
/* prox!(y, ψ, q_or_g = q, sigma), else iprox!(y, ψ, q_or_g = g, d) */
typedef struct spx_box_job_f64 {
  int32_t op;
  int32_t reserved;
  double* y_host;
  const double* q_or_g_host;
  const double* d_host;
  double lambda, sigma;
} spx_box_job_f64;
typedef struct spx_box_job_f32 {
  int32_t op;
  int32_t reserved;
  float* y_host;
  const float* q_or_g_host;
  const float* d_host;
  double lambda, sigma;
} spx_box_job_f32;

#define SPX_DECL_SEPARABLE(SUF, R)                                                               \
  /* ShiftedNormL1.prox!  shiftedNormL1.jl:40-54 */                                              \
  int32_t spx_prox_l1_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q, \
                            double lambda, double sigma, double* psi_out);                       \
  /* ShiftedNormL1.iprox! shiftedNormL1.jl:60-75; first_bad_d (host, may be NULL): index of  */ \
  /* the first d[i] <= 0 or -1; when given the call synchronises and returns SPX_E_ASSERT_D */  \
  int32_t spx_iprox_l1_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,            \
                             const R* g, const R* d, double lambda, int64_t* first_bad_d,        \
                             double* psi_out);                                                   \
  /* ShiftedNormL0.prox!  shiftedNormL0.jl:38-55 */                                              \
  int32_t spx_prox_l0_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q, \
                            double lambda, double sigma, double* psi_out);                       \
  /* ShiftedNormL0.iprox! shiftedNormL0.jl:61-80 */                                              \
  int32_t spx_iprox_l0_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,            \
                             const R* g, const R* d, double lambda, int64_t* first_bad_d,        \
                             double* psi_out);                                                   \
  /* ShiftedRootNormLhalf.prox! shiftedRootNormLhalf.jl:41-63 (ψ.sol is not materialised). */    \
  /* xk == sj == NULL: the unshifted RootNormLhalf.prox!(y, h, x = q, γ = sigma) of */           \
  /* rootNormLhalf.jl:31-51; psi_out then receives its return value h(y). */                     \
  int32_t spx_prox_lhalf_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,          \
                               const R* q, double lambda, double sigma, double* psi_out);        \
  /* ---------------------------------------------------- Box / BInf (a8-a12) */                 \
  /* ShiftedNormL1Box.prox!  shiftedNormL1Box.jl:89-125 */                                       \
  int32_t spx_prox_l1box_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,          \
                               const R* q, const spx_bound* l, const spx_bound* u,               \
                               const spx_sel* sel, double lambda, double sigma,                  \
                               double* psi_out);                                                 \
  /* ShiftedNormL1Box.iprox! shiftedNormL1Box.jl:131-225 */                                      \
  int32_t spx_iprox_l1box_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,         \
                                const R* g, const R* d, const spx_bound* l, const spx_bound* u,  \
                                const spx_sel* sel, double lambda, double* psi_out);             \
  /* ShiftedNormL0Box.prox!  shiftedNormL0Box.jl:89-131 */                                       \
  int32_t spx_prox_l0box_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,          \
                               const R* q, const spx_bound* l, const spx_bound* u,               \
                               const spx_sel* sel, double lambda, double sigma,                  \
                               double* psi_out);                                                 \
  /* ShiftedNormL0Box.iprox! shiftedNormL0Box.jl:137-231 (a NaN g[i] with |d[i]| < eps, */      \
  /* where the reference leaves y[i] untouched, yields NaN here: y is write-only) */            \
  int32_t spx_iprox_l0box_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,         \
                                const R* g, const R* d, const spx_bound* l, const spx_bound* u,  \
                                const spx_sel* sel, double lambda, double* psi_out);             \
  /* ShiftedRootNormLhalfBox.prox! shiftedRootNormLhalfBox.jl:86-120 */                          \
  int32_t spx_prox_lhalfbox_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,       \
                                  const R* q, const spx_bound* l, const spx_bound* u,            \
                                  const spx_sel* sel, double lambda, double sigma,               \
                                  double* psi_out);                                              \
  /* ---------------------------------------------------- ShiftedNormL1B2 (a13) */               \
  /* ShiftedNormL1B2.prox! shiftedNormL1B2.jl:47-64.  chi_lambda is χ.lambda (NormL2(1.0) */    \
  /* in the reference's tests).  passes_out (host, may be NULL): number of vector passes. */    \
  int32_t spx_prox_l1b2_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,           \
                              const R* q, double lambda, double sigma, double delta,             \
                              double chi_lambda, int32_t* passes_out, double* psi_out);          \
  /* the same prox! on this rank's contiguous shard of a vector sharded over several GPUs: */   \
  /* the K partial sums of squares of every pass (and the two ψ sums) go through `reduce`; */   \
  /* the scalar root search is replicated, so every rank takes identical decisions */           \
  int32_t spx_prox_l1b2_sharded_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,   \
                                      const R* q, double lambda, double sigma, double delta,     \
                                      double chi_lambda, spx_allreduce_sum_fn reduce,            \
                                      void* user, int32_t* passes_out, double* psi_out);         \
  /* building blocks (one pass each), exported for tests: */                                     \
  /* sumsq_out[k] = Σ_i ProjB(-xk_i * scale[k])_i^2, k < nscale <= 16 (host arrays); */        \
  /* scale == NULL -> the unscaled ProjB(-xk) of :56 */                                          \
  int32_t spx_l1b2_projnorm2_##SUF(spx_ctx* ctx, int64_t n, const R* xk, const R* sj,            \
                                   const R* q, double lambda, double sigma, int32_t nscale,      \
                                   const double* scale_host, double* sumsq_out_host);            \
  /* y = ProjB(-xk * scale) * post - sj  (:60-62); use_scale = 0 -> y = ProjB(-xk) - sj */      \
  int32_t spx_l1b2_finish_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,         \
                                const R* q, double lambda, double sigma, int32_t use_scale,      \
                                double scale, double post, double delta, double* psi_sum_out,    \
                                double* w_sumsq_out);                                            \
  /* ------------------------------------------------------ group norms (a14-a15) */             \
  /* ShiftedGroupNormL2.prox! shiftedGroupNormL2.jl:52-79; groups are contiguous index */       \
  /* ranges offs[g]..offs[g+1]-1 (device int64, ngroups+1 entries), lambda_g device R[ngroups] */\
  /* xk == sj == NULL (prox_groupl2 only): the unshifted GroupNormL2.prox!(y, h, x = q, γ = sigma) of */ \
  /* groupNormL2.jl:41-58; psi_out then receives its return value Σ_g λ_g ‖x_g‖ (input norms). */ \
  int32_t spx_prox_groupl2_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,        \
                                 const R* q, int64_t ngroups, const int64_t* offs,               \
                                 const R* lambda_g, double sigma, double* psi_out);              \
  /* ShiftedGroupNormL2Binf.prox! shiftedGroupNormL2Binf.jl:67-119 */                            \
  int32_t spx_prox_groupl2binf_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,    \
                                     const R* q, int64_t ngroups, const int64_t* offs,           \
                                     const R* lambda_g, double sigma, double delta,              \
                                     double* psi_out);                                           \
  /* ------------------------------------------------------ top-r (a16-a17) */                   \
  /* ShiftedIndBallL0.prox! shiftedIndBallL0.jl:54-72 and ShiftedIndBallL0BInf.prox! */         \
  /* shiftedIndBallL0BInf.jl:73-95 (binf != 0 -> clamp to ±delta).  nprob independent */        \
  /* problems of length n stored back to back (nprob = 1 for a single ψ).  The `p` */           \
  /* permutation scratch of the reference does not exist: radix-select, no sort. */             \
  int32_t spx_prox_indballl0_##SUF(spx_ctx* ctx, int64_t nprob, int64_t n, R* y, const R* xk,    \
                                   const R* sj, const R* q, int64_t r, int32_t binf,             \
                                   double delta);                                                \
  /* one vector spread over `world` GPUs in rank order (this rank holds n_local contiguous elements of */ \
  /* the n_global): the 2048-bin histogram of every radix digit goes through `reduce` (sum over ranks), */ \
  /* then one vector of `world` tie counts; lowest global index wins ties, as on one GPU.  reduce == NULL: */ \
  /* the context's communicator (spx_comm_init, `world` ranks) all-reduces histograms and tie counts on */    \
  /* the device, with no host staging */                                                                   \
  int32_t spx_prox_indballl0_sharded_##SUF(spx_ctx* ctx, int64_t n_local, int64_t n_global, R* y,       \
                                           const R* xk, const R* sj, const R* q, int64_t r,            \
                                           int32_t binf, double delta, int32_t rank, int32_t world,    \
                                           spx_allreduce_sum_fn reduce, void* user);                   \
  /* ------------------------------------------------------ ψ(y) (a18-a20) */                    \
  /* generic ψ(y) = h(xk + sj + y), ShiftedProximalOperators.jl:51-54; kind = SPX_H_L1, */      \
  /* _L0, _LHALF, _INDBALLL0 (param r) */                                                        \
  int32_t spx_value_sep_##SUF(spx_ctx* ctx, int32_t kind, int64_t n, const R* xk, const R* sj,   \
                              const R* y, double lambda, int64_t r, double* out);                \
  /* Box ψ(y): shiftedNormL1Box.jl:70-82, shiftedNormL0Box.jl:70-82, */                          \
  /* shiftedRootNormLhalfBox.jl:67-79 */                                                         \
  int32_t spx_value_box_##SUF(spx_ctx* ctx, int32_t kind, int64_t n, const R* xk, const R* sj,   \
                              const R* y, const spx_bound* l, const spx_bound* u,                \
                              const spx_sel* sel, double lambda, double* out);                   \
  /* ShiftedNormL1B2 ψ(y): shiftedNormL1B2.jl:32 */                                              \
  int32_t spx_value_l1b2_##SUF(spx_ctx* ctx, int64_t n, const R* xk, const R* sj, const R* y,    \
                               double lambda, double delta, double* out);                        \
  /* BInf ψ(y): shiftedIndBallL0BInf.jl:44-49 (kind SPX_H_INDBALLL0) and */                      \
  /* shiftedGroupNormL2Binf.jl:34-39 (kind SPX_H_GROUPL2) */                                     \
  int32_t spx_value_binf_##SUF(spx_ctx* ctx, int32_t kind, int64_t n, const R* xk, const R* sj,  \
                               const R* y, double delta, int64_t r, int64_t ngroups,             \
                               const int64_t* offs, const R* lambda_g, double* out);             \
  /* ShiftedGroupNormL2 ψ(y): ShiftedProximalOperators.jl:51-54 + groupNormL2.jl:33-39 */        \
  int32_t spx_value_groupl2_##SUF(spx_ctx* ctx, int64_t n, const R* xk, const R* sj,             \
                                  const R* y, int64_t ngroups, const int64_t* offs,              \
                                  const R* lambda_g, double* out);                               \
  /* partial sums for sharded vectors: out_host[0] = Σ (un-scaled by λ), out_host[1] = 1.0 */   \
  /* if the shard is infeasible; the caller all-reduces (sum, max) and applies λ / Inf */       \
  int32_t spx_value_partial_##SUF(spx_ctx* ctx, int32_t kind, int64_t n, const R* xk,            \
                                  const R* sj, const R* y, const spx_bound* l,                   \
                                  const spx_bound* u, const spx_sel* sel, int32_t boxed,         \
                                  double* out_host);                                             \
  /* ------------------------------ fused solver step (SURVEY.md §8f rank 1) */                 \
  /* The sweeps a solver iteration wraps around every prox! (R2 / TR of RegularizedOptimization.jl,          */ \
  /* reference README.md:17) or iprox! (R2DH / TRDH), in one call:                                           */ \
  /*   q = (-nu) .* grad   (spx_step_*)    rounded to R like the caller's broadcast                          */ \
  /*   d = D .+ dshift     (spx_istep_*)   rounded to R likewise                                             */ \
  /*   s = prox!(ψ, q, nu) or iprox!(ψ, grad, d)   [the method bodies cited at spx_prox_* / spx_iprox_*]     */ \
  /*   xsy = (xk + sj) + s                         [ψ's argument, ShiftedProximalOperators.jl:52;            */ \
  /*                                                xsy == NULL: not written]                                */ \
  /*   out3_host = {ψ(s), Σ s_i², Σ grad_i s_i}    [ψ(s): ShiftedProximalOperators.jl:51-54, Inf outside     */ \
  /*                                                the type's box or ball]                                  */ \
  /*   out4_host = out3_host and Σ d_i s_i²        (spx_istep_*)                                             */ \
  /* The sums are in Float64.  s is bit for bit the type's spx_prox_* of that q with sigma = nu (spx_iprox_* */ \
  /* of grad and that d).  sj == NULL reads as zeros (ψ shifted once) for spx_step_sep / _box and            */ \
  /* spx_istep_*; the other steps need sj (zeros when ψ is shifted once).  Every step synchronises, and      */ \
  /* its scalars are all-reduced when the context reduces scalars.                                           */ \
  /* Aliasing, for n > 0: no output (s, xsy) overlaps an input (xk, sj, grad, D, l->vec, u->vec) or the      */ \
  /* other output partially, and beyond that (anything else: SPX_E_INVALID)                                  */ \
  /*                                   s == grad   s == xk or sj   xsy == an input or s                      */ \
  /*   spx_step_sep / _box, istep_*    yes         yes             yes                                       */ \
  /*   groupl2, groupl2binf, indballl0 no          no              yes                                       */ \
  /*   l1b2, l1b2_sharded              no          yes             yes, but xsy must not overlap s           */ \
  /* The one-pass forms read every element's (group's) operands before they write its results.  The          */ \
  /* composed forms below write q into s before prox! reads xk and sj, and spx_step_post reads grad;         */ \
  /* the search of spx_step_l1b2 keeps its stash in s while the finish writes xsy.                           */ \
  /* kind = SPX_H_L1, _L0, _LHALF: one pass                                                                  */ \
  int32_t spx_step_sep_##SUF(spx_ctx* ctx, int32_t kind, int64_t n, R* s, R* xsy, const R* xk,   \
                             const R* sj, const R* grad, double lambda, double nu,               \
                             double* out3_host);                                                 \
  /* the Box / BInf forms; op: 0 L1Box, 1 L0Box, 2 LhalfBox: one pass                                        */ \
  int32_t spx_step_box_##SUF(spx_ctx* ctx, int32_t op, int64_t n, R* s, R* xsy, const R* xk,     \
                             const R* sj, const R* grad, const spx_bound* l, const spx_bound* u, \
                             const spx_sel* sel, double lambda, double nu, double* out3_host);   \
  /* kind = SPX_H_L1, _L0 (no iprox! for _LHALF: SPX_E_INVALID): one pass.  The `@assert d[i] > 0` of the    */ \
  /* unboxed forms applies to d: SPX_E_ASSERT_D and *first_bad_d (may be NULL) as for spx_iprox_l1; s is     */ \
  /* written in full either way.                                                                             */ \
  int32_t spx_istep_sep_##SUF(spx_ctx* ctx, int32_t kind, int64_t n, R* s, R* xsy, const R* xk,  \
                              const R* sj, const R* grad, const R* D, double dshift,             \
                              double lambda, int64_t* first_bad_d, double* out4_host);           \
  /* the Box forms; op: 0 L1Box, 1 L0Box (2 LhalfBox: SPX_E_INVALID): one pass                               */ \
  int32_t spx_istep_box_##SUF(spx_ctx* ctx, int32_t op, int64_t n, R* s, R* xsy, const R* xk,    \
                              const R* sj, const R* grad, const R* D, double dshift,             \
                              const spx_bound* l, const spx_bound* u, const spx_sel* sel,        \
                              double lambda, double* out4_host);                                 \
  /* The composed form of the step around a prox! that is not one streaming pass (groups, top-r): the        */ \
  /* caller's sweeps as two passes around the type's own entry point --                                      */ \
  /*   spx_step_pre:   q = (-nu) .* grad (rounded to R), written where s will be;                            */ \
  /*   the type's spx_prox_* IN PLACE (y = q = s, sigma = nu, its psi_out / value entry gives ψ(s));         */ \
  /*   spx_step_post:  xsy = (xk + sj) + s (xsy may be NULL), out2_host = {Σ s², Σ grad·s}.                  */ \
  /* sj == NULL: zeros.  spx_step_post synchronises.                                                         */ \
  int32_t spx_step_pre_##SUF(spx_ctx* ctx, int64_t n, R* q, const R* grad, double nu);               \
  /* ShiftedGroupNormL2 (shiftedGroupNormL2.jl:52-79): on every layout, inside the passes of the prox!      */ \
  /* kernels of its group sizes -- ONE pass per group (two grid-wide passes for a single group spanning the  */ \
  /* vector), no spx_step_pre / spx_step_post.  A layout rewritten after validation is still computed right: */ \
  /* only the groups the first kernel left are read again, so xsy may alias xk or sj in that case as well.  */ \
  int32_t spx_step_groupl2_##SUF(spx_ctx* ctx, int64_t n, R* s, R* xsy, const R* xk, const R* sj,    \
                                 const R* grad, int64_t ngroups, const int64_t* offs,                \
                                 const R* lambda_g, double nu, double* out3_host);                   \
  /* ShiftedGroupNormL2Binf (shiftedGroupNormL2Binf.jl:67-119): ONE pass when the layout is uniform          */ \
  /* (n == ngroups m, m in {16, 32, 64, 128, 256}, offs == {0, m, 2m, ...}, ngroups > 1, 16-byte aligned     */ \
  /* vectors), the composed form otherwise.  ψ(s) of shiftedGroupNormL2Binf.jl:34-39: Inf when sj + s        */ \
  /* leaves the ball of 1.1 delta.                                                                           */ \
  int32_t spx_step_groupl2binf_##SUF(spx_ctx* ctx, int64_t n, R* s, R* xsy, const R* xk,             \
                                     const R* sj, const R* grad, int64_t ngroups,                    \
                                     const int64_t* offs, const R* lambda_g, double nu,              \
                                     double delta, double* out3_host);                               \
  /* ShiftedIndBallL0 (shiftedIndBallL0.jl:54-72) and ShiftedIndBallL0BInf (binf != 0,                       */ \
  /* shiftedIndBallL0BInf.jl:73-95) for nprob problems of length n back to back: ONE pass of the stream      */ \
  /* top-r kernel when spx_prox_indballl0 would take its stream form (16-byte aligned vectors, n % 8 == 0,   */ \
  /* 4096 <= n <= 131072, 0 < r < n, nprob >= 2 x the SM count) and xsy is given and overlaps no input,      */ \
  /* the composed form otherwise.  ψ(s) as the type's ψ(y) returns it over the whole batch (the count of     */ \
  /* xk + sj + s != 0 against r; BInf: Inf when sj + s leaves the ball of 1.1 delta,                         */ \
  /* shiftedIndBallL0BInf.jl:44-49).                                                                         */ \
  int32_t spx_step_indballl0_##SUF(spx_ctx* ctx, int64_t nprob, int64_t n, R* s, R* xsy,             \
                                   const R* xk, const R* sj, const R* grad, int64_t r, int32_t binf, \
                                   double delta, double nu, double* out3_host);                      \
  /* ShiftedNormL1B2 (shiftedNormL1B2.jl:47-64) inside the passes of its own root search: every pass         */ \
  /* forms q on the load, the finish writes s and xsy.  ψ(s) as psi_out of spx_prox_l1b2 (λ Σ|xk + sj + s|   */ \
  /* rounded to R, Inf when ‖sj + s‖ leaves the ball of delta, shiftedNormL1B2.jl:32); passes_out (may be    */ \
  /* NULL) as for spx_prox_l1b2.  s uses itself as scratch, and the finish doubles as the check of an        */ \
  /* unverified root, only when s and xsy overlap none of xk, sj, grad; otherwise (xsy = xk: x <- x + s)     */ \
  /* the search converges by evaluation and each element's operands are read before its results are          */ \
  /* written.  Every decision of the search is all-reduced when the context reduces scalars.                 */ \
  int32_t spx_step_l1b2_##SUF(spx_ctx* ctx, int64_t n, R* s, R* xsy, const R* xk, const R* sj,       \
                              const R* grad, double lambda, double nu, double delta,                 \
                              double chi_lambda, int32_t* passes_out, double* out3_host);            \
  /* the same step on this rank's shard of a sharded vector: `reduce` gets the 2K partial sums of            */ \
  /* every norm pass and, once, the finish's four {Σ|xk + sj + s|, Σ (sj + s)², Σ s², Σ grad·s}              */ \
  int32_t spx_step_l1b2_sharded_##SUF(spx_ctx* ctx, int64_t n, R* s, R* xsy, const R* xk,            \
                                      const R* sj, const R* grad, double lambda, double nu,          \
                                      double delta, double chi_lambda, spx_allreduce_sum_fn reduce,  \
                                      void* user, int32_t* passes_out, double* out3_host);           \
  int32_t spx_step_post_##SUF(spx_ctx* ctx, int64_t n, R* xsy, const R* xk, const R* sj, const R* s, \
                              const R* grad, double* out2_host);                                     \
  /* ------------------------------ host-buffer entry points (end-to-end path) */              \
  /* Box prox!/iprox! with every vector in HOST memory (pinned for full speed): chunked, */     \
  /* H2D / kernel / D2H overlapped on three streams.  op: 0 L1Box, 1 L0Box, 2 LhalfBox; */      \
  /* gd_host == NULL -> prox!(q_or_g = q, sigma); else iprox!(q_or_g = g, d)  */                \
  int32_t spx_box_host_##SUF(spx_ctx* ctx, int32_t op, int64_t n, R* y_host, const R* xk_host,   \
                             const R* sj_host, const R* q_or_g_host, const R* d_host,            \
                             const R* l_host, double l_val, const R* u_host, double u_val,       \
                             double lambda, double sigma, int64_t chunk_elems,                   \
                             double* psi_out);                                                   \
  /* Several Box prox!/iprox! at the SAME shifted point (xk, sj, l, u) in one pass over the */   \
  /* host vectors: each chunk of xk, sj, l, u and of every distinct q/g/d vector crosses PCIe */ \
  /* once, the nops kernels run back to back on it, and the nops outputs travel back while */    \
  /* the next chunk is uploaded.  This is the solver-side pattern (several regularizers / */    \
  /* a prox! and an iprox! evaluated at one iterate).  Host vectors named by several ops are */  \
  /* recognised by pointer.  psi_out: NULL or nops doubles (ψ(y) of each op).  */                \
  int32_t spx_box_multi_host_##SUF(spx_ctx* ctx, int32_t nops, const spx_box_job_##SUF* jobs,    \
                                   int64_t n, const R* xk_host, const R* sj_host,                \
                                   const R* l_host, double l_val, const R* u_host, double u_val, \
                                   int64_t chunk_elems, double* psi_out);

SPX_DECL_SEPARABLE(f64, double)
SPX_DECL_SEPARABLE(f32, float)

/* ---- thresholding stage of the spectral operators, GIVEN an SVD (SURVEY.md §8f rank 4) ----------------------------
 * ShiftedRank / ShiftedNuclearnorm / ShiftedCappedl1 prox! (shiftedRank.jl:68-84, shiftedNuclearnorm.jl:68-81,
 * shiftedCappedl1.jl:68-86):  sol = q + xk + sj;  U, S, Vt = svd(reshape(sol));  S' = threshold(S);  U[:, i] *= S'_i;
 * A = U * Vt;  y = reshape(A) - (xk + sj).  The SVD (LAPACK in the reference) and the GEMM (`mul!`) stay library
 * calls on the caller's side (cuSOLVER / cuBLAS); these three entry points are the stages around them.
 *   kind 0 Rank:        column i zeroed where S_i <= sqrt(2 lambda sigma), scaled by S_i elsewhere (S untouched)
 *   kind 1 Nuclearnorm: S_i = max(0, S_i - lambda sigma), column scaled by it
 *   kind 2 Cappedl1:    S_i = the better of max(theta, S_i) and min(theta, max(0, S_i - lambda sigma)) (:72-77)
 * u: m x k column-major, leading dimension ldu; s: k singular values (overwritten for kinds 1, 2 like ψ.h.F.S). */
#define SPX_SPECTRAL_RANK 0
#define SPX_SPECTRAL_NUCLEAR 1
#define SPX_SPECTRAL_CAPPEDL1 2
#define SPX_DECL_SPECTRAL(SUF, R)                                                                               \
  /* a_out = (q + xk) + sj   (`ψ.sol .= q .+ ψ.xk .+ ψ.sj`, shiftedRank.jl:69) */                               \
  int32_t spx_spectral_sol_##SUF(spx_ctx* ctx, int64_t n, R* a_out, const R* xk, const R* sj, const R* q);     \
  int32_t spx_spectral_threshold_##SUF(spx_ctx* ctx, int32_t kind, int64_t m, int64_t k, R* u, int64_t ldu,    \
                                       R* s, double lambda, double sigma, double theta);                       \
  /* y = a - (xk + sj)   (shiftedRank.jl:82) */                                                                 \
  int32_t spx_spectral_finish_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* a, const R* xk, const R* sj);
SPX_DECL_SPECTRAL(f64, double)
SPX_DECL_SPECTRAL(f32, float)

/* scalar helpers, exported for the glue's unit tests:
 * prox_zero  ShiftedProximalOperators.jl:203, iprox_zero :217-236 */
double spx_prox_zero_f64(double q, double l, double u);
double spx_iprox_zero_f64(double d, double g, double l, double u);
float spx_prox_zero_f32(float q, float l, float u);
float spx_iprox_zero_f32(float d, float g, float l, float u);

#ifdef __cplusplus
}
#endif
#endif /* SHIFTEDPROX_H */
