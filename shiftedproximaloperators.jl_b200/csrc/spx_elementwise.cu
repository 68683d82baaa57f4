// spx_elementwise.cu -- C entry points of the separable / Box prox!, iprox! and ψ(y).
#include "spx_elementwise.cuh"
#include "spx_ops.cuh"
#include "spx_setup.cuh"

namespace spx {

#define SPX_CHECK_VEC3(ctx, n, y, a, b, c)                                   \
  SPX_REQUIRE((ctx) != nullptr, "null context");                             \
  SPX_REQUIRE((n) >= 0, "n < 0");                                            \
  SPX_REQUIRE((n) == 0 || ((y) && (a) && (b) && (c)), "null device vector"); \
  DeviceGuard guard__((ctx)->device)

// run op (with or without fused ψ), optionally fold and return the value
template <template <class, bool> class OpT, class R, class Setup>
static int32_t run_sep(spx_ctx* ctx, int64_t n, int kind, R lambda, double* psi_out, Setup setup) {
  if (psi_out == nullptr) {
    OpT<R, false> op;
    setup(op);
    return ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, nullptr);
  }
  OpT<R, true> op;
  setup(op);
  int nb = 0;
  int32_t st = ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, &nb);
  if (st != SPX_OK) return st;
  st = finalize_partials(ctx, nb, 1, false);
  if (st != SPX_OK) return st;
  *psi_out = scale_value<R>(kind, lambda, ctx->h_result[0].s, 0);
  return SPX_OK;
}

template <class R>
static int32_t prox_l1(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q, double lambda,
                       double sigma, double* psi_out) {
  SPX_CHECK_VEC3(ctx, n, y, xk, sj, q);
  const R lam = (R)lambda, sig = (R)sigma;
  return run_sep<ProxL1, R>(ctx, n, SPX_H_L1, lam, psi_out, [&](auto& op) {
    set3(op, xk, sj, q);
    op.y = y;
    configure(op, lam, sig);
  });
}

template <class R>
static int32_t prox_l0(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q, double lambda,
                       double sigma, double* psi_out) {
  SPX_CHECK_VEC3(ctx, n, y, xk, sj, q);
  const R lam = (R)lambda, sig = (R)sigma;
  return run_sep<ProxL0, R>(ctx, n, SPX_H_L0, lam, psi_out, [&](auto& op) {
    set3(op, xk, sj, q);
    op.y = y;
    configure(op, lam, sig);
  });
}

template <class R>
static int32_t prox_lhalf(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q, double lambda,
                          double sigma, double* psi_out) {
  // xk == sj == NULL: the unshifted RootNormLhalf prox! (rootNormLhalf.jl:31-51), shifts read as zeros
  SPX_REQUIRE(ctx != nullptr, "null context");
  SPX_REQUIRE(n >= 0, "n < 0");
  SPX_REQUIRE(n == 0 || (y && q), "null device vector");
  SPX_REQUIRE((xk == nullptr) == (sj == nullptr), "xk and sj must both be given or both be NULL");
  DeviceGuard guard__(ctx->device);
  const R lam = (R)lambda, sig = (R)sigma;
  return run_sep<ProxLhalf, R>(ctx, n, SPX_H_LHALF, lam, psi_out, [&](auto& op) {
    set3(op, xk, sj, q);
    op.y = y;
    configure(op, lam, sig);
  });
}

// iprox! of the unboxed L1 / L0: the assertion flag always travels with the pass
template <template <class, bool> class OpT, class R>
static int32_t iprox_sep(spx_ctx* ctx, int kind, int64_t n, R* y, const R* xk, const R* sj, const R* g, const R* d,
                         double lambda, int64_t* first_bad_d, double* psi_out) {
  SPX_CHECK_VEC3(ctx, n, y, xk, sj, g);
  SPX_REQUIRE(n == 0 || d != nullptr, "null d");
  const R lam = (R)lambda;
  auto setup = [&](auto& op) { set_iprox(op, y, xk, sj, g, d, lam); };
  int nb = 0;
  int32_t st;
  if (psi_out) {
    OpT<R, true> op;
    setup(op);
    st = ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, &nb);
  } else {
    OpT<R, false> op;
    setup(op);
    st = ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, &nb);
  }
  if (st != SPX_OK) return st;
  if (first_bad_d == nullptr && psi_out == nullptr) return SPX_OK;  // asynchronous, unchecked
  st = finalize_partials(ctx, nb, 1, false);
  if (st != SPX_OK) return st;
  if (psi_out) *psi_out = scale_value<R>(kind, lam, ctx->h_result[0].s, 0);
  long long bad = ctx->h_result[0].bad;
  long long idx = bad < 0 ? -1 : ((1ll << 62) - bad);
  if (first_bad_d) *first_bad_d = idx;
  if (idx >= 0) {
    set_error("AssertionError: d[%lld] > 0", idx);
    return SPX_E_ASSERT_D;
  }
  return SPX_OK;
}

// --------------------------------------------------------------------- Box --
template <class R, bool PSI>
static int32_t launch_box_t(spx_ctx* ctx, cudaStream_t stream, int opc, bool inverse, int64_t n, R* y, const R* xk,
                            const R* sj, const R* qg, const R* d, const R* lvec, R lval, const R* uvec, R uval,
                            DevSel sel, R lambda, R sigma, Partial* partials, int* nb, int64_t base) {
  if (!inverse) {
    if (opc == BOX_L1) {
      ProxL1Box<R, PSI> op;
      set_box(op, xk, sj, qg, d, lvec, lval, uvec, uval);
      op.y = y; op.sel = sel;
      configure(op, lambda, sigma);
      return ew_launch(ctx, stream, op, n, base, partials, nb);
    } else if (opc == BOX_L0) {
      ProxL0Box<R, PSI> op;
      set_box(op, xk, sj, qg, d, lvec, lval, uvec, uval);
      op.y = y; op.sel = sel;
      configure(op, lambda, sigma);
      return ew_launch(ctx, stream, op, n, base, partials, nb);
    } else if (opc == BOX_LHALF) {
      ProxLhalfBox<R, PSI> op;
      set_box(op, xk, sj, qg, d, lvec, lval, uvec, uval);
      op.y = y; op.sel = sel;
      configure(op, lambda, sigma);
      return ew_launch(ctx, stream, op, n, base, partials, nb);
    }
  } else {
    if (opc == BOX_L1) {
      IproxL1Box<R, PSI> op;
      set_iprox_box(op, y, xk, sj, qg, d, lvec, lval, uvec, uval, sel, lambda);
      return ew_launch(ctx, stream, op, n, base, partials, nb);
    } else if (opc == BOX_L0) {
      IproxL0Box<R, PSI> op;
      set_iprox_box(op, y, xk, sj, qg, d, lvec, lval, uvec, uval, sel, lambda);
      return ew_launch(ctx, stream, op, n, base, partials, nb);
    }
  }
  set_error("unknown Box operator %d (inverse=%d)", opc, (int)inverse);
  return SPX_E_INVALID;
}

template <class R>
int32_t launch_box(spx_ctx* ctx, cudaStream_t stream, int op, bool inverse, int64_t n, R* y, const R* xk, const R* sj,
                   const R* qg, const R* d, const R* lvec, R lval, const R* uvec, R uval, DevSel sel, R lambda,
                   R sigma, bool want_psi, Partial* partials, int* nblocks_out, int64_t index_base) {
  if (want_psi)
    return launch_box_t<R, true>(ctx, stream, op, inverse, n, y, xk, sj, qg, d, lvec, lval, uvec, uval, sel, lambda,
                                 sigma, partials, nblocks_out, index_base);
  return launch_box_t<R, false>(ctx, stream, op, inverse, n, y, xk, sj, qg, d, lvec, lval, uvec, uval, sel, lambda,
                                sigma, partials, nblocks_out, index_base);
}
template int32_t launch_box<double>(spx_ctx*, cudaStream_t, int, bool, int64_t, double*, const double*, const double*,
                                    const double*, const double*, const double*, double, const double*, double, DevSel,
                                    double, double, bool, Partial*, int*, int64_t);
template int32_t launch_box<float>(spx_ctx*, cudaStream_t, int, bool, int64_t, float*, const float*, const float*,
                                   const float*, const float*, const float*, float, const float*, float, DevSel, float,
                                   float, bool, Partial*, int*, int64_t);

template <class R>
static int32_t box_entry(spx_ctx* ctx, int opc, bool inverse, int64_t n, R* y, const R* xk, const R* sj, const R* qg,
                         const R* d, const spx_bound* l, const spx_bound* u, const spx_sel* sel, double lambda,
                         double sigma, double* psi_out) {
  SPX_CHECK_VEC3(ctx, n, y, xk, sj, qg);
  SPX_REQUIRE(l && u, "null bounds");
  SPX_REQUIRE(!inverse || n == 0 || d != nullptr, "null d");
  DevSel ds;
  int32_t st = make_sel(sel, n, &ds);
  if (st != SPX_OK) return st;
  int nb = 0;
  st = launch_box<R>(ctx, ctx->stream, opc, inverse, n, y, xk, sj, qg, d, (const R*)l->vec, (R)l->val,
                     (const R*)u->vec, (R)u->val, ds, (R)lambda, (R)sigma, psi_out != nullptr, ctx->d_partials, &nb, 0);
  if (st != SPX_OK || psi_out == nullptr) return st;
  st = finalize_partials(ctx, nb, 1, false);
  if (st != SPX_OK) return st;
  *psi_out = ctx->h_result[0].bad > 0 ? kInf : scale_value<R>(box_kind(opc), (R)lambda, ctx->h_result[0].s, 0);
  return SPX_OK;
}

// ------------------------------------------------------------------ values --
template <class R>
static int32_t value_sep(spx_ctx* ctx, int32_t kind, int64_t n, const R* xk, const R* sj, const R* y, double lambda,
                         int64_t r, double* out) {
  SPX_CHECK_VEC3(ctx, n, out, xk, sj, y);
  SPX_REQUIRE(kind >= SPX_H_L1 && kind <= SPX_H_INDBALLL0, "unknown h kind");
  ValueSep<R> op;
  set3(op, xk, sj, y);
  op.y = nullptr;
  op.kind = kind;
  int nb = 0;
  int32_t st = ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, &nb);
  if (st != SPX_OK) return st;
  st = finalize_partials(ctx, nb, 1, false);
  if (st != SPX_OK) return st;
  *out = scale_value<R>(kind, (R)lambda, ctx->h_result[0].s, r);
  return SPX_OK;
}

// gather over an explicit `selected` list (duplicates count twice: shiftedNormL1Box.jl:71)
template <class R>
__global__ void __launch_bounds__(256) gather_value_kernel(int kind, const long long* __restrict__ list,
                                                           long long nlist, long long n, const R* __restrict__ xk,
                                                           const R* __restrict__ sj, const R* __restrict__ y,
                                                           Partial* __restrict__ partials) {
  Partial acc;
  acc.s = 0.0; acc.s2 = 0.0; acc.bad = -1;
  for (long long j = (long long)blockIdx.x * 256 + threadIdx.x; j < nlist; j += (long long)gridDim.x * 256) {
    long long i = list[j];
    if (i >= 0 && i < n) acc.s += h_term(kind, (xk[i] + sj[i]) + y[i]);
  }
  acc = block_fold<256>(acc);
  if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}

// raw (Σ, infeasible) of a Box / plain ψ(y) over one shard
template <class R>
static int32_t value_raw(spx_ctx* ctx, int32_t kind, int64_t n, const R* xk, const R* sj, const R* y,
                         const spx_bound* l, const spx_bound* u, const spx_sel* sel, bool boxed, double* sum,
                         bool* infeasible) {
  *sum = 0.0;
  *infeasible = false;
  int nb = 0;
  int32_t st;
  if (!boxed) {
    ValueSep<R> op;
    set3(op, xk, sj, y);
    op.y = nullptr;
    op.kind = kind;
    st = ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, &nb);
    if (st != SPX_OK) return st;
    st = finalize_partials(ctx, nb, 1, false);
    if (st != SPX_OK) return st;
    *sum = ctx->h_result[0].s;
    return SPX_OK;
  }
  DevSel ds;
  st = make_sel(sel, n, &ds);
  if (st != SPX_OK) return st;
  const bool use_list = sel != nullptr && sel->list != nullptr && sel->kind != SPX_SEL_ALL;
  ValueBox<R> op;
  op.in[0] = xk; op.in[1] = sj; op.in[2] = y;
  op.in[3] = (const R*)l->vec; op.in[4] = (const R*)u->vec;
  op.fill[0] = op.fill[1] = op.fill[2] = R(0);
  op.fill[3] = (R)l->val; op.fill[4] = (R)u->val;
  op.y = nullptr;
  op.sel = ds;
  op.kind = kind;
  op.weigh = !use_list;
  st = ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, &nb);
  if (st != SPX_OK) return st;
  st = finalize_partials(ctx, nb, 1, false);
  if (st != SPX_OK) return st;
  *sum = ctx->h_result[0].s;
  *infeasible = ctx->h_result[0].bad > 0;
  if (use_list) {
    long long want = (sel->nlist + 255) / 256;
    if (want < 1) want = 1;
    int grid = (int)(want < (long long)ctx->sm_count * 8 ? want : (long long)ctx->sm_count * 8);
    gather_value_kernel<R><<<grid, 256, 0, ctx->stream>>>(kind, (const long long*)sel->list, sel->nlist, n, xk, sj, y,
                                                          ctx->d_partials);
    ctx->launches++;
    SPX_CUDA(cudaGetLastError());
    st = finalize_partials(ctx, grid, 1, false);
    if (st != SPX_OK) return st;
    *sum = ctx->h_result[0].s;
  }
  return SPX_OK;
}

template <class R>
static int32_t value_box(spx_ctx* ctx, int32_t kind, int64_t n, const R* xk, const R* sj, const R* y,
                         const spx_bound* l, const spx_bound* u, const spx_sel* sel, double lambda, double* out) {
  SPX_CHECK_VEC3(ctx, n, out, xk, sj, y);
  SPX_REQUIRE(l && u, "null bounds");
  SPX_REQUIRE(kind >= SPX_H_L1 && kind <= SPX_H_LHALF, "unknown h kind");
  double sum;
  bool inf;
  int32_t st = value_raw<R>(ctx, kind, n, xk, sj, y, l, u, sel, true, &sum, &inf);
  if (st != SPX_OK) return st;
  *out = inf ? kInf : scale_value<R>(kind, (R)lambda, sum, 0);
  return SPX_OK;
}

template <class R>
static int32_t value_partial(spx_ctx* ctx, int32_t kind, int64_t n, const R* xk, const R* sj, const R* y,
                             const spx_bound* l, const spx_bound* u, const spx_sel* sel, int32_t boxed, double* out) {
  SPX_CHECK_VEC3(ctx, n, out, xk, sj, y);
  SPX_REQUIRE(!boxed || (l && u), "null bounds");
  SPX_REQUIRE(kind >= SPX_H_L1 && kind <= SPX_H_INDBALLL0, "unknown h kind");
  double sum;
  bool inf;
  int32_t st = value_raw<R>(ctx, kind, n, xk, sj, y, l, u, sel, boxed != 0, &sum, &inf);
  if (st != SPX_OK) return st;
  out[0] = sum;
  out[1] = inf ? 1.0 : 0.0;
  return SPX_OK;
}

// IndBallL2(Δ) of ProximalOperators 0.15: 0 iff ‖w‖ ≤ Δ or isapprox(‖w‖, Δ; atol=eps, rtol=√eps)
template <class R> static bool in_ball_l2(R nw, R delta) {
  const R eps = std::numeric_limits<R>::epsilon();
  if (nw <= delta) return true;
  if (!std::isfinite(nw) || !std::isfinite(delta)) return false;
  R tol = std::max(eps, std::sqrt(eps) * std::max(std::fabs(nw), std::fabs(delta)));
  return std::fabs(nw - delta) <= tol;
}

template <class R>
static int32_t value_l1b2(spx_ctx* ctx, int64_t n, const R* xk, const R* sj, const R* y, double lambda, double delta,
                          double* out) {
  SPX_CHECK_VEC3(ctx, n, out, xk, sj, y);
  ValueL1B2<R> op;
  set3(op, xk, sj, y);
  op.y = nullptr;
  int nb = 0;
  int32_t st = ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, &nb);
  if (st != SPX_OK) return st;
  st = finalize_partials(ctx, nb, 1, false);
  if (st != SPX_OK) return st;
  R nw = (R)std::sqrt(ctx->h_result[0].s2);
  *out = in_ball_l2<R>(nw, (R)delta) ? scale_value<R>(SPX_H_L1, (R)lambda, ctx->h_result[0].s, 0) : kInf;
  return SPX_OK;
}

// group part lives in spx_group.cu
template <class R>
int32_t value_group_binf(spx_ctx* ctx, int64_t n, const R* xk, const R* sj, const R* y, bool binf, double delta,
                         int64_t ngroups, const int64_t* offs, const R* lambda_g, double* out);

template <class R>
static int32_t value_binf(spx_ctx* ctx, int32_t kind, int64_t n, const R* xk, const R* sj, const R* y, double delta,
                          int64_t r, int64_t ngroups, const int64_t* offs, const R* lambda_g, double* out) {
  SPX_CHECK_VEC3(ctx, n, out, xk, sj, y);
  if (kind == SPX_H_GROUPL2) return value_group_binf<R>(ctx, n, xk, sj, y, true, delta, ngroups, offs, lambda_g, out);
  SPX_REQUIRE(kind == SPX_H_INDBALLL0, "BInf value: kind must be INDBALLL0 or GROUPL2");
  ValueBinfCount<R> op;
  set3(op, xk, sj, y);
  op.y = nullptr;
  op.rad = 1.1 * (double)(R)delta;
  int nb = 0;
  int32_t st = ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, &nb);
  if (st != SPX_OK) return st;
  st = finalize_partials(ctx, nb, 1, false);
  if (st != SPX_OK) return st;
  double hv = ctx->h_result[0].s <= (double)r ? 0.0 : kInf;
  *out = ctx->h_result[0].bad > 0 ? kInf : hv;
  return SPX_OK;
}

}  // namespace spx

using namespace spx;

#define SPX_DEFINE_EW(SUF, R)                                                                                     \
  extern "C" int32_t spx_prox_l1_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q,       \
                                       double lambda, double sigma, double* psi_out) {                            \
    return prox_l1<R>(ctx, n, y, xk, sj, q, lambda, sigma, psi_out);                                              \
  }                                                                                                               \
  extern "C" int32_t spx_iprox_l1_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* g,      \
                                        const R* d, double lambda, int64_t* first_bad_d, double* psi_out) {       \
    return iprox_sep<IproxL1, R>(ctx, SPX_H_L1, n, y, xk, sj, g, d, lambda, first_bad_d, psi_out);                \
  }                                                                                                               \
  extern "C" int32_t spx_prox_l0_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q,       \
                                       double lambda, double sigma, double* psi_out) {                            \
    return prox_l0<R>(ctx, n, y, xk, sj, q, lambda, sigma, psi_out);                                              \
  }                                                                                                               \
  extern "C" int32_t spx_iprox_l0_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* g,      \
                                        const R* d, double lambda, int64_t* first_bad_d, double* psi_out) {       \
    return iprox_sep<IproxL0, R>(ctx, SPX_H_L0, n, y, xk, sj, g, d, lambda, first_bad_d, psi_out);                \
  }                                                                                                               \
  extern "C" int32_t spx_prox_lhalf_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q,    \
                                          double lambda, double sigma, double* psi_out) {                         \
    return prox_lhalf<R>(ctx, n, y, xk, sj, q, lambda, sigma, psi_out);                                           \
  }                                                                                                               \
  extern "C" int32_t spx_prox_l1box_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q,    \
                                          const spx_bound* l, const spx_bound* u, const spx_sel* sel,             \
                                          double lambda, double sigma, double* psi_out) {                         \
    return box_entry<R>(ctx, BOX_L1, false, n, y, xk, sj, q, nullptr, l, u, sel, lambda, sigma, psi_out);         \
  }                                                                                                               \
  extern "C" int32_t spx_iprox_l1box_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* g,   \
                                           const R* d, const spx_bound* l, const spx_bound* u,                    \
                                           const spx_sel* sel, double lambda, double* psi_out) {                  \
    return box_entry<R>(ctx, BOX_L1, true, n, y, xk, sj, g, d, l, u, sel, lambda, 0.0, psi_out);                  \
  }                                                                                                               \
  extern "C" int32_t spx_prox_l0box_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q,    \
                                          const spx_bound* l, const spx_bound* u, const spx_sel* sel,             \
                                          double lambda, double sigma, double* psi_out) {                         \
    return box_entry<R>(ctx, BOX_L0, false, n, y, xk, sj, q, nullptr, l, u, sel, lambda, sigma, psi_out);         \
  }                                                                                                               \
  extern "C" int32_t spx_iprox_l0box_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* g,   \
                                           const R* d, const spx_bound* l, const spx_bound* u,                    \
                                           const spx_sel* sel, double lambda, double* psi_out) {                  \
    return box_entry<R>(ctx, BOX_L0, true, n, y, xk, sj, g, d, l, u, sel, lambda, 0.0, psi_out);                  \
  }                                                                                                               \
  extern "C" int32_t spx_prox_lhalfbox_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,             \
                                             const R* q, const spx_bound* l, const spx_bound* u,                  \
                                             const spx_sel* sel, double lambda, double sigma, double* psi_out) {  \
    return box_entry<R>(ctx, BOX_LHALF, false, n, y, xk, sj, q, nullptr, l, u, sel, lambda, sigma, psi_out);      \
  }                                                                                                               \
  extern "C" int32_t spx_value_sep_##SUF(spx_ctx* ctx, int32_t kind, int64_t n, const R* xk, const R* sj,         \
                                         const R* y, double lambda, int64_t r, double* out) {                     \
    return value_sep<R>(ctx, kind, n, xk, sj, y, lambda, r, out);                                                 \
  }                                                                                                               \
  extern "C" int32_t spx_value_box_##SUF(spx_ctx* ctx, int32_t kind, int64_t n, const R* xk, const R* sj,         \
                                         const R* y, const spx_bound* l, const spx_bound* u, const spx_sel* sel,  \
                                         double lambda, double* out) {                                            \
    return value_box<R>(ctx, kind, n, xk, sj, y, l, u, sel, lambda, out);                                         \
  }                                                                                                               \
  extern "C" int32_t spx_value_l1b2_##SUF(spx_ctx* ctx, int64_t n, const R* xk, const R* sj, const R* y,          \
                                          double lambda, double delta, double* out) {                             \
    return value_l1b2<R>(ctx, n, xk, sj, y, lambda, delta, out);                                                  \
  }                                                                                                               \
  extern "C" int32_t spx_value_binf_##SUF(spx_ctx* ctx, int32_t kind, int64_t n, const R* xk, const R* sj,        \
                                          const R* y, double delta, int64_t r, int64_t ngroups,                   \
                                          const int64_t* offs, const R* lambda_g, double* out) {                  \
    return value_binf<R>(ctx, kind, n, xk, sj, y, delta, r, ngroups, offs, lambda_g, out);                        \
  }                                                                                                               \
  extern "C" int32_t spx_value_partial_##SUF(spx_ctx* ctx, int32_t kind, int64_t n, const R* xk, const R* sj,     \
                                             const R* y, const spx_bound* l, const spx_bound* u,                  \
                                             const spx_sel* sel, int32_t boxed, double* out_host) {               \
    return value_partial<R>(ctx, kind, n, xk, sj, y, l, u, sel, boxed, out_host);                                 \
  }

SPX_DEFINE_EW(f64, double)
SPX_DEFINE_EW(f32, float)

// ------------------------------------------------------------------ self-test --
namespace spx {
__device__ __forceinline__ unsigned long long st_mix(unsigned long long x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
// random double with a uniformly random mantissa and an exponent in [-emax, emax]
__device__ __forceinline__ double st_rand(unsigned long long h, int emax) {
  const unsigned long long mant = h & 0x000fffffffffffffull;
  const int e = (int)((h >> 52) % (unsigned)(2 * emax + 1)) - emax;
  const double m = __longlong_as_double((long long)(mant | 0x3ff0000000000000ull));
  return ldexp(m, e) * ((h >> 63) ? -1.0 : 1.0);
}
__global__ void __launch_bounds__(256) selftest_kernel(long long n, unsigned long long seed,
                                                       unsigned long long* __restrict__ bad) {
  unsigned long long b0 = 0, b1 = 0, b2 = 0;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const unsigned long long h1 = st_mix(seed + 3 * (unsigned long long)i);
    const unsigned long long h2 = st_mix(seed + 3 * (unsigned long long)i + 1);
    const unsigned long long h3 = st_mix(seed + 3 * (unsigned long long)i + 2);
    const double x = fabs(st_rand(h1, 60)), a = st_rand(h2, 40), d = st_rand(h3, 40);
    if (__double_as_longlong(sqrt_fast(x)) != __double_as_longlong(sqrt(x))) ++b0;
    const Quot3<double> q = quot3(a, d, 1.0 + fabs(x), true);
    const Quot3<double> r = quot3_ref<double>(a, d, 1.0 + fabs(x));
    if (__double_as_longlong(q.a) != __double_as_longlong(r.a) || __double_as_longlong(q.b) != __double_as_longlong(r.b) ||
        __double_as_longlong(q.c) != __double_as_longlong(r.c))
      ++b1;
    const double s = 0.05 + fabs(ldexp(d, -ilogb(d)));  // divisor of order 1
    if (__double_as_longlong(div_uniform(a, s, 1.0 / s)) != __double_as_longlong(a / s)) ++b2;
  }
  if (b0) atomicAdd(bad + 0, b0);
  if (b1) atomicAdd(bad + 1, b1);
  if (b2) atomicAdd(bad + 2, b2);
}
}  // namespace spx

extern "C" int32_t spx_selftest_math(spx_ctx* ctx, int64_t n, uint64_t seed, int64_t* mismatches_out) {
  SPX_REQUIRE(ctx && mismatches_out, "null argument");
  SPX_REQUIRE(n >= 0, "n < 0");
  DeviceGuard g(ctx->device);
  int32_t st = ensure_scratch(ctx, 4096);
  if (st != SPX_OK) return st;
  SPX_CUDA(cudaMemsetAsync(ctx->d_scratch, 0, 24, ctx->stream));
  if (n > 0) {
    selftest_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(n, seed, (unsigned long long*)ctx->d_scratch);
    ctx->launches++;
    SPX_CUDA(cudaGetLastError());
  }
  SPX_CUDA(cudaMemcpyAsync(mismatches_out, ctx->d_scratch, 24, cudaMemcpyDeviceToHost, ctx->stream));
  SPX_CUDA(cudaStreamSynchronize(ctx->stream));
  return SPX_OK;
}
