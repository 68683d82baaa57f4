// spx_step.cu -- the fused solver step (SURVEY.md §8f rank 1).
//
// The callers of the shifted prox (the R2 / TR inner iterations of RegularizedOptimization.jl, reference
// README.md:17) surround every prox! with sweeps over the same vectors:
//     mν∇f .= -ν .* ∇f;  prox!(s, ψ, mν∇f, ν);  ψ(s);  xk + s;  ‖s‖;  ∇f's
// -- 15 vector transits for what needs 4 (read xk, ∇f; write s, xk+s).  One pass here does all of it:
//     q_i   = (-ν) ∇f_i                      (rounded to R like the caller's broadcast)
//     s_i   = prox!(ψ, q, ν)_i               the functors of spx_ops.cuh, bit for bit the stand-alone prox!
//     xsy_i = (xk_i + sj_i) + s_i            ψ's own argument (ShiftedProximalOperators.jl:52), optional output
//     ψ(s)  = h(xsy) [+ Inf outside the box] (ShiftedProximalOperators.jl:51-54, shiftedNormL1Box.jl:70-82)
//     Σ s_i²,  Σ ∇f_i s_i                    in Float64
// Same streaming structure as ew_kernel (spx_elementwise.cuh): 128-bit loads of every operand, UNROLL
// independent requests per stream before the first use, streaming stores, one partial slot per CTA folded
// in fixed order.
//
// The diagonal quasi-Newton iterations (R2DH, TRDH) wrap iprox!(s, ψ, ∇f, D .+ σ) in the same sweeps plus the model's
// quadratic term; the iprox! form of the kernel (IPROX) does that step in the same pass:
//     d_i   = D_i + σ                        (rounded to R like the caller's broadcast)
//     s_i   = iprox!(ψ, ∇f, d)_i             IproxL1/L0 and their Box forms, bit for bit the stand-alone iprox!
//     xsy_i, ψ(s), Σ s_i², Σ ∇f_i s_i        as above,  and  Σ d_i s_i²  in Float64
#include "spx_elementwise.cuh"
#include "spx_ops.cuh"
#include "spx_setup.cuh"

namespace spx {

// resident CTAs per SM: the step carries two more accumulators and a second output row than the prox! alone,
// so the Box functors (which ask for 4 CTAs = 64 registers) get 3 CTAs = 84 registers and do not spill
#ifndef SPX_STEP_MINB
#define SPX_STEP_MINB 3
#endif
// The iprox! form also keeps d, ∇f and Σ d s² live.  Under the 84 registers of 3 CTAs the Float64 IproxL0Box instance
// spills 36 bytes, so that form alone gets 2 CTAs = 128 registers.  The other Box forms keep 3: on a B200 at n = 2^28
// Float64 / 2^29 Float32 they ran about 3 % faster there than at 2 (profiles/r05_istep_ops_ctas.txt).
template <class Op> struct IstepTwoCtas : std::false_type {};
template <bool PSI> struct IstepTwoCtas<IproxL0Box<double, PSI>> : std::true_type {};
template <class Op, bool IPROX = false> struct StepBlocks {
  static constexpr int cap = IPROX && IstepTwoCtas<Op>::value ? 2 : SPX_STEP_MINB;
  static constexpr int value = MinBlocks<Op>::value > cap ? cap : MinBlocks<Op>::value;
};

// An operator whose ψ fills both accumulators of the first slot (L1B2StepFinish: Σ|xk+sj+s| and Σ(sj+s)²) declares
// SUMSQ_SLOT1: Σs² then goes to the second slot's s2, beside Σ∇f·s.
template <class Op, class = void> struct SumsqSlot1 { static constexpr bool value = false; };
template <class Op> struct SumsqSlot1<Op, std::void_t<decltype(Op::SUMSQ_SLOT1)>> {
  static constexpr bool value = Op::SUMSQ_SLOT1;
};

// IPROX = false: the step around prox!, c = -ν scales ∇f into q.
// IPROX = true:  the step around iprox!, ∇f goes to the functor as loaded, c = σ shifts the diagonal (x[3]) into
//                d = D + σ, and Σ d s² is summed as well.
template <int VEC, int UNROLL, class Op, bool IPROX = false>
__global__ void __launch_bounds__(kEwThreads, StepBlocks<Op, IPROX>::value)
    step_kernel(const Op op, const typename Op::Real c, typename Op::Real* xsy, const long long n,
                Partial* __restrict__ partials) {
  using R = typename Op::Real;
  constexpr int NIN = Op::NIN;
  Partial acc;
  acc.s = 0.0;
  acc.s2 = 0.0;
  acc.bad = -1;
  double dot = 0.0, sds = 0.0;
  auto element = [&](R (&x)[NIN], long long i, R& s, R& v) {
    const R g = x[2];
    if constexpr (IPROX)
      x[3] = x[3] + c;  // d = D + σ
    else
      x[2] = c * g;  // q = -ν ∇f
    s = op.apply(x, i, acc);
    v = (x[0] + x[1]) + s;
    if constexpr (SumsqSlot1<Op>::value)
      sds = __fma_rn((double)s, (double)s, sds);
    else
      acc.s2 = __fma_rn((double)s, (double)s, acc.s2);
    dot = __fma_rn((double)g, (double)s, dot);
    if constexpr (IPROX) sds = __fma_rn((double)x[3] * (double)s, (double)s, sds);
  };

  const long long nvec = n / VEC;
  const long long tile = (long long)kEwThreads * UNROLL;
  for (long long base = (long long)blockIdx.x * tile; base < nvec; base += (long long)gridDim.x * tile) {
    Pack<R, VEC> reg[NIN][UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const long long v = base + (long long)u * kEwThreads + threadIdx.x;
#pragma unroll
      for (int k = 0; k < NIN; ++k) {
        if (op.in[k] != nullptr && v < nvec) {
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
        Pack<R, VEC> out, out2;
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
          R x[NIN];
#pragma unroll
          for (int k = 0; k < NIN; ++k) x[k] = reg[k][u].v[e];
          element(x, v * VEC + e, out.v[e], out2.v[e]);
        }
        st_stream(op.y + v * VEC, out);
        if (xsy != nullptr) st_stream(xsy + v * VEC, out2);
      }
    }
  }
  if (VEC > 1 && blockIdx.x == gridDim.x - 1) {  // scalar tail
    const long long i = nvec * VEC + threadIdx.x;
    if (i < n) {
      R x[NIN], s, v;
#pragma unroll
      for (int k = 0; k < NIN; ++k) x[k] = op.in[k] != nullptr ? op.in[k][i] : op.fill[k];
      element(x, i, s, v);
      op.y[i] = s;
      if (xsy != nullptr) xsy[i] = v;
    }
  }
  acc = block_fold<kEwThreads>(acc);
  Partial second;
  second.s = dot;
  second.s2 = sds;
  second.bad = -1;
  second = block_fold<kEwThreads>(second);
  if (threadIdx.x == 0) {
    partials[blockIdx.x] = acc;
    partials[gridDim.x + blockIdx.x] = second;
  }
}

template <int VEC, int UNROLL, class Op, bool IPROX> static int step_blocks_per_sm() {
  static int cached = 0;  // per instantiation
  if (cached == 0) {
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, step_kernel<VEC, UNROLL, Op, IPROX>, kEwThreads, 0) !=
            cudaSuccess ||
        nb < 1)
      nb = 1;
    cached = nb;
  }
  return cached;
}

// launch and fold the two slots into ctx->h_result: [0] = (ψ sum, Σs², flag), [1] = (Σ∇f·s, Σ d s² or 0);
// SUMSQ_SLOT1 operators: [0] = (their two ψ sums), [1] = (Σ∇f·s, Σs²)
template <bool IPROX, class Op, class R>
static int32_t step_launch(spx_ctx* ctx, const Op& op, R c, R* xsy, int64_t n) {
  constexpr int VECW = 16 / (int)sizeof(R);
  constexpr int UNROLL = Op::UNROLL;
  int nb = 0;
  if (n > 0) {
    bool vec = aligned16(op) && (((uintptr_t)xsy) & 15u) == 0;
    const long long nvec = vec ? n / VECW : n;
    const long long tile = (long long)kEwThreads * UNROLL;
    long long want = (nvec + tile - 1) / tile;
    if (want < 1) want = 1;
    long long cap = (long long)ctx->sm_count * (vec ? step_blocks_per_sm<VECW, UNROLL, Op, IPROX>()
                                                    : step_blocks_per_sm<1, UNROLL, Op, IPROX>());
    if (cap > kMaxPartials) cap = kMaxPartials;
    nb = (int)(want < cap ? want : cap);
    if (vec)
      step_kernel<VECW, UNROLL, Op, IPROX><<<nb, kEwThreads, 0, ctx->stream>>>(op, c, xsy, n, ctx->d_partials);
    else
      step_kernel<1, UNROLL, Op, IPROX><<<nb, kEwThreads, 0, ctx->stream>>>(op, c, xsy, n, ctx->d_partials);
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "step_kernel launch");
  }
  return finalize_partials(ctx, nb, 2, false);
}

// the step around prox!: hand back (ψ(s), Σs², Σ∇f·s)
template <class Op, class R>
static int32_t step_run(spx_ctx* ctx, const Op& op, R nu, R* xsy, int64_t n, int kind, R lambda, double* out3) {
  int32_t st = step_launch<false>(ctx, op, -nu, xsy, n);
  if (st != SPX_OK) return st;
  out3[0] = ctx->h_result[0].bad > 0 ? kInf : scale_value<R>(kind, lambda, ctx->h_result[0].s, 0);
  out3[1] = ctx->h_result[0].s2;
  out3[2] = ctx->h_result[1].s;
  return SPX_OK;
}

#define SPX_STEP_COMMON_CHECKS()                                                   \
  SPX_REQUIRE(ctx != nullptr, "null context");                                     \
  SPX_REQUIRE(n >= 0, "n < 0");                                                    \
  SPX_REQUIRE(out3 != nullptr, "null result array");                               \
  SPX_REQUIRE(n == 0 || (s && xk && grad), "null device vector");                  \
  DeviceGuard guard__(ctx->device)

template <class R>
static int32_t step_sep(spx_ctx* ctx, int32_t kind, int64_t n, R* s, R* xsy, const R* xk, const R* sj, const R* grad,
                        double lambda, double nu, double* out3) {
  SPX_STEP_COMMON_CHECKS();
  const R lam = (R)lambda, sig = (R)nu;
  auto go = [&](auto op) {
    set3(op, xk, sj, grad);
    op.y = s;
    configure(op, lam, sig);
    return step_run(ctx, op, sig, xsy, n, kind, lam, out3);
  };
  if (kind == SPX_H_L1) return go(ProxL1<R, true>{});
  if (kind == SPX_H_L0) return go(ProxL0<R, true>{});
  if (kind == SPX_H_LHALF) return go(ProxLhalf<R, true>{});
  set_error("spx_step_sep: h kind %d has no separable prox!", (int)kind);
  return SPX_E_INVALID;
}

template <class R>
static int32_t step_box(spx_ctx* ctx, int32_t opc, int64_t n, R* s, R* xsy, const R* xk, const R* sj, const R* grad,
                        const spx_bound* l, const spx_bound* u, const spx_sel* sel, double lambda, double nu,
                        double* out3) {
  SPX_STEP_COMMON_CHECKS();
  SPX_REQUIRE(l && u, "null bounds");
  DevSel ds;
  int32_t st = make_sel(sel, n, &ds);
  if (st != SPX_OK) return st;
  const R lam = (R)lambda, sig = (R)nu;
  auto go = [&](auto op) {
    set_box(op, xk, sj, grad, (const R*)nullptr, (const R*)l->vec, (R)l->val, (const R*)u->vec, (R)u->val);
    op.y = s;
    op.sel = ds;
    configure(op, lam, sig);
    return step_run(ctx, op, sig, xsy, n, box_kind(opc), lam, out3);
  };
  if (opc == BOX_L1) return go(ProxL1Box<R, true>{});
  if (opc == BOX_L0) return go(ProxL0Box<R, true>{});
  if (opc == BOX_LHALF) return go(ProxLhalfBox<R, true>{});
  set_error("spx_step_box: unknown Box operator %d", (int)opc);
  return SPX_E_INVALID;
}

// ---- the step around iprox! (diagonal model: R2DH, TRDH) --------------------------------------------------------
// The same pass with the iprox! functors: d = D + σ in R, s = iprox!(ψ, ∇f, d), and out4 = (ψ(s), Σs², Σ∇f·s, Σ d s²).
#define SPX_ISTEP_COMMON_CHECKS()                                                  \
  SPX_REQUIRE(ctx != nullptr, "null context");                                     \
  SPX_REQUIRE(n >= 0, "n < 0");                                                    \
  SPX_REQUIRE(out4 != nullptr, "null result array");                               \
  SPX_REQUIRE(n == 0 || (s && xk && grad && D), "null device vector");             \
  DeviceGuard guard__(ctx->device)

static void istep_sums(const spx_ctx* ctx, double* out4) {
  out4[1] = ctx->h_result[0].s2;
  out4[2] = ctx->h_result[1].s;
  out4[3] = ctx->h_result[1].s2;
}

template <class R>
static int32_t istep_sep(spx_ctx* ctx, int32_t kind, int64_t n, R* s, R* xsy, const R* xk, const R* sj, const R* grad,
                         const R* D, double dshift, double lambda, int64_t* first_bad_d, double* out4) {
  SPX_ISTEP_COMMON_CHECKS();
  const R lam = (R)lambda;
  auto go = [&](auto op) {
    set_iprox(op, s, xk, sj, grad, D, lam);
    int32_t st = step_launch<true>(ctx, op, (R)dshift, xsy, n);
    if (st != SPX_OK) return st;
    out4[0] = scale_value<R>(kind, lam, ctx->h_result[0].s, 0);
    istep_sums(ctx, out4);
    const long long bad = ctx->h_result[0].bad;  // first d[i] <= 0, as in iprox_sep (spx_elementwise.cu)
    const long long idx = bad < 0 ? -1 : ((1ll << 62) - bad);
    if (first_bad_d) *first_bad_d = idx;
    if (idx >= 0) {
      set_error("AssertionError: d[%lld] > 0", idx);
      return SPX_E_ASSERT_D;
    }
    return SPX_OK;
  };
  if (kind == SPX_H_L1) return go(IproxL1<R, true>{});
  if (kind == SPX_H_L0) return go(IproxL0<R, true>{});
  set_error("spx_istep_sep: h kind %d has no iprox!", (int)kind);
  return SPX_E_INVALID;
}

template <class R>
static int32_t istep_box(spx_ctx* ctx, int32_t opc, int64_t n, R* s, R* xsy, const R* xk, const R* sj, const R* grad,
                         const R* D, double dshift, const spx_bound* l, const spx_bound* u, const spx_sel* sel,
                         double lambda, double* out4) {
  SPX_ISTEP_COMMON_CHECKS();
  SPX_REQUIRE(l && u, "null bounds");
  if (opc != BOX_L1 && opc != BOX_L0) {
    set_error("spx_istep_box: Box operator %d has no iprox!", (int)opc);
    return SPX_E_INVALID;
  }
  DevSel ds;
  int32_t st = make_sel(sel, n, &ds);
  if (st != SPX_OK) return st;
  const R lam = (R)lambda;
  auto go = [&](auto op) {
    set_iprox_box(op, s, xk, sj, grad, D, (const R*)l->vec, (R)l->val, (const R*)u->vec, (R)u->val, ds, lam);
    int32_t st = step_launch<true>(ctx, op, (R)dshift, xsy, n);
    if (st != SPX_OK) return st;
    out4[0] = ctx->h_result[0].bad > 0 ? kInf : scale_value<R>(box_kind(opc), lam, ctx->h_result[0].s, 0);
    istep_sums(ctx, out4);
    return SPX_OK;
  };
  return opc == BOX_L1 ? go(IproxL1Box<R, true>{}) : go(IproxL0Box<R, true>{});
}

// ---- the step around a prox! that is not one streaming pass (groups, top-r, ShiftedNormL1B2) ----------------------
// The caller's sweeps collapse into two passes around the operator's own kernels:
//   pre:   q = (-ν) ∇f  written where s will be (the prox! then runs in place: prox!(s, ψ, s, ν));
//   post:  xsy = (xk + sj) + s,  Σ s²,  Σ ∇f·s   in one pass (ψ(s) comes from the prox! / ψ(y) entry of the type).
// 1R + 1W and 4R + 1W next to the operator, instead of the caller's 11 transits for the same sweeps.
template <class R> struct StepPre {
  using Real = R;
  static constexpr int NIN = 1, UNROLL = 4;
  static constexpr bool OUT = true, ACC = false;
  const R* in[NIN];  // ∇f
  R fill[NIN];
  R* y;
  R mnu;
  __device__ __forceinline__ R apply(const R (&x)[NIN], long long, Partial&) const { return mnu * x[0]; }
};
template <class R, bool WRITE> struct StepPost {
  using Real = R;
  static constexpr int NIN = 4, UNROLL = 2;
  static constexpr bool OUT = WRITE, ACC = true;
  const R* in[NIN];  // xk, sj (NULL: zeros), s, ∇f
  R fill[NIN];
  R* y;  // xsy
  __device__ __forceinline__ R apply(const R (&x)[NIN], long long, Partial& acc) const {
    acc.s2 = __fma_rn((double)x[2], (double)x[2], acc.s2);
    acc.s = __fma_rn((double)x[3], (double)x[2], acc.s);
    return (x[0] + x[1]) + x[2];
  }
};

template <class R> int32_t step_pre(spx_ctx* ctx, int64_t n, R* q, const R* grad, double nu) {
  SPX_REQUIRE(ctx != nullptr, "null context");
  SPX_REQUIRE(n >= 0, "n < 0");
  SPX_REQUIRE(n == 0 || (q && grad), "null device vector");
  DeviceGuard guard(ctx->device);
  StepPre<R> op;
  op.in[0] = grad;
  op.fill[0] = R(0);
  op.y = q;
  op.mnu = -(R)nu;
  int nb = 0;
  return ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, &nb);
}
template <class R>
int32_t step_post(spx_ctx* ctx, int64_t n, R* xsy, const R* xk, const R* sj, const R* s, const R* grad, double* out2) {
  SPX_REQUIRE(ctx != nullptr, "null context");
  SPX_REQUIRE(n >= 0, "n < 0");
  SPX_REQUIRE(out2 != nullptr, "null result array");
  SPX_REQUIRE(n == 0 || (xk && s && grad), "null device vector");
  DeviceGuard guard(ctx->device);
  int nb = 0;
  auto go = [&](auto op) {
    op.in[0] = xk; op.in[1] = sj; op.in[2] = s; op.in[3] = grad;
    op.fill[0] = op.fill[1] = op.fill[2] = op.fill[3] = R(0);
    op.y = xsy;
    return ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, &nb);
  };
  int32_t st = xsy ? go(StepPost<R, true>{}) : go(StepPost<R, false>{});
  if (st != SPX_OK) return st;
  st = finalize_partials(ctx, nb, 1, false);
  if (st != SPX_OK) return st;
  out2[0] = ctx->h_result[0].s2;
  out2[1] = ctx->h_result[0].s;
  return SPX_OK;
}

// The finish pass of the ShiftedNormL1B2 step's root search (spx_l1b2.cu): s = ProjB(-xk scale) post - sj with
// q = (-ν)∇f, xsy = (xk + sj) + s (xsy may be NULL), and v = {Σ|xk+sj+s|, Σ(sj+s)², Σs², Σ∇f·s}.  mid: the search's
// stash of sj + q (it is s itself), NULL when there is none.  Its grid is step_kernel's, not the prox! finish's
// (ew_kernel): where the two differ, Σ(sj+s)² -- and with it the check of an unverified root -- is summed in another order.
template <class R>
int32_t step_l1b2_finish(spx_ctx* ctx, int64_t n, R* s, R* xsy, const R* xk, const R* sj, const R* grad, const R* mid,
                         R nu, R ls, bool use_scale, R scale, R post, double* v) {
  L1B2StepFinish<R> op;
  op.in[0] = xk; op.in[1] = sj; op.in[2] = grad; op.in[3] = mid;
  op.fill[0] = op.fill[1] = op.fill[2] = op.fill[3] = R(0);
  op.y = s;
  op.f = L1B2Finish<R, true>{};
  op.f.ls = ls; op.f.scale = scale; op.f.post = post; op.f.use_scale = use_scale;
  op.f.have_mid = mid != nullptr;
  int32_t st = step_launch<false>(ctx, op, -nu, xsy, n);
  if (st != SPX_OK) return st;
  v[0] = ctx->h_result[0].s;
  v[1] = ctx->h_result[0].s2;
  v[2] = ctx->h_result[1].s2;
  v[3] = ctx->h_result[1].s;
  return SPX_OK;
}

template int32_t step_l1b2_finish<double>(spx_ctx*, int64_t, double*, double*, const double*, const double*,
                                          const double*, const double*, double, double, bool, double, double, double*);
template int32_t step_l1b2_finish<float>(spx_ctx*, int64_t, float*, float*, const float*, const float*, const float*,
                                         const float*, float, float, bool, float, float, double*);
template int32_t step_pre<double>(spx_ctx*, int64_t, double*, const double*, double);
template int32_t step_pre<float>(spx_ctx*, int64_t, float*, const float*, double);
template int32_t step_post<double>(spx_ctx*, int64_t, double*, const double*, const double*, const double*, const double*,
                                   double*);
template int32_t step_post<float>(spx_ctx*, int64_t, float*, const float*, const float*, const float*, const float*,
                                  double*);

}  // namespace spx

using namespace spx;

#define SPX_DEFINE_STEP(SUF, R)                                                                                       \
  extern "C" int32_t spx_step_sep_##SUF(spx_ctx* ctx, int32_t kind, int64_t n, R* s, R* xsy, const R* xk,             \
                                        const R* sj, const R* grad, double lambda, double nu, double* out3) {         \
    return step_sep<R>(ctx, kind, n, s, xsy, xk, sj, grad, lambda, nu, out3);                                         \
  }                                                                                                                   \
  extern "C" int32_t spx_step_box_##SUF(spx_ctx* ctx, int32_t op, int64_t n, R* s, R* xsy, const R* xk, const R* sj,  \
                                        const R* grad, const spx_bound* l, const spx_bound* u, const spx_sel* sel,    \
                                        double lambda, double nu, double* out3) {                                     \
    return step_box<R>(ctx, op, n, s, xsy, xk, sj, grad, l, u, sel, lambda, nu, out3);                                \
  }                                                                                                                   \
  extern "C" int32_t spx_step_pre_##SUF(spx_ctx* ctx, int64_t n, R* q, const R* grad, double nu) {                    \
    return step_pre<R>(ctx, n, q, grad, nu);                                                                          \
  }                                                                                                                   \
  extern "C" int32_t spx_step_post_##SUF(spx_ctx* ctx, int64_t n, R* xsy, const R* xk, const R* sj, const R* s,       \
                                         const R* grad, double* out2) {                                               \
    return step_post<R>(ctx, n, xsy, xk, sj, s, grad, out2);                                                          \
  }                                                                                                                   \
  extern "C" int32_t spx_istep_sep_##SUF(spx_ctx* ctx, int32_t kind, int64_t n, R* s, R* xsy, const R* xk,            \
                                         const R* sj, const R* grad, const R* D, double dshift, double lambda,        \
                                         int64_t* first_bad_d, double* out4) {                                        \
    return istep_sep<R>(ctx, kind, n, s, xsy, xk, sj, grad, D, dshift, lambda, first_bad_d, out4);                    \
  }                                                                                                                   \
  extern "C" int32_t spx_istep_box_##SUF(spx_ctx* ctx, int32_t op, int64_t n, R* s, R* xsy, const R* xk, const R* sj, \
                                         const R* grad, const R* D, double dshift, const spx_bound* l,                \
                                         const spx_bound* u, const spx_sel* sel, double lambda, double* out4) {       \
    return istep_box<R>(ctx, op, n, s, xsy, xk, sj, grad, D, dshift, l, u, sel, lambda, out4);                        \
  }

SPX_DEFINE_STEP(f64, double)
SPX_DEFINE_STEP(f32, float)
