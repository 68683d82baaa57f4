// spx_l1b2.cu -- ShiftedNormL1B2 prox!  (shiftedNormL1B2.jl:47-64).
//
//   ProjB(z) = min(max(z, sj+q-λσ), sj+q+λσ);  y = ProjB(-xk)
//   if Δ <= χ(y):  η = root of η - χ(ProjB(-xk η/Δ));  y = ProjB(-xk η/Δ) Δ/η
//   y -= sj
//
// Every evaluation of the residual is a full streaming pass over xk, sj, q (3R per element; 2R once
// mid = sj + q has been stashed in the output vector, which the search is free to use as scratch when it
// aliases no input), so the pass count is what matters.  A pass evaluates up to 4 trial values of η at once and
// returns, next to Σw², the sum Σ w dw/dη that gives the derivative of the residual (~12 instructions per trial:
// four trials keep the pass HBM-bound, eight are FP64-issue bound).  Roots' one-point-per-pass iteration becomes:
// a ladder pass Δ·{1, 2, 4, 16} (its first value decides whether the ball is active), then clusters of four trial
// values around the root of the cubic Hermite interpolant of the residual on the bracket, and the finish pass as
// the check of the last interpolated root (see prox_l1b2 below): 3 norm passes + finish on large vectors.  End
// state: a point with |residual| <= 4 ulp, an exact zero, or -- as Roots' bisection -- two adjacent floats around
// the sign change.  When the vector is sharded over several GPUs the partial sums of every pass are all-reduced, by
// the context's communicator (spx_comm.cu) or by the caller's callback; the scalar search is replicated on every rank.
#include <algorithm>
#include <cstring>
#include <vector>

#include "spx_elementwise.cuh"
#include "spx_ops.cuh"

namespace spx {

template <int K> struct ScaleSet { double s[K]; };
#ifndef SPX_L1B2_UNROLL
#define SPX_L1B2_UNROLL 2
#endif
// Packets loaded per thread and trip before the first use.  Float64: two (a 2R pass keeps only 32 B per thread in
// flight otherwise).  Float32: two only in the single-trial pass (the decision pass -- all there is when the ball
// is inactive); with four trials a Float32 packet already carries 16 element-trials of arithmetic per 16 bytes and
// the second packet's registers spill.  Measured: Float64 n = 2^28 7.34 -> 6.64 ms; Float32 n = 2^29 active
// 7.47 -> 7.99 ms with two packets everywhere, inactive 2.49 -> 2.38 ms.
template <class R, int K> struct L1b2Unroll {
  static constexpr int value = sizeof(R) == 8 ? SPX_L1B2_UNROLL : (K == 1 ? SPX_L1B2_UNROLL : 1);
  static constexpr int minb = (value > 1 && sizeof(R) == 8 && K <= 4) ? 4 : 1;  // resident CTAs asked of ptxas
};

// Σ_i ProjB(z_i(k))² and Σ_i ProjB(z_i(k)) dProjB/dscale (= Σ over the unclamped entries of z_i (-xk_i))
// for K scalings in one pass.  The clamp is two compares and selects (a NaN z stays NaN; a NaN bound is
// caught by the `mid - mid` poison term, so a NaN anywhere still makes every norm NaN like Base.min/max).
// MODE 0: mid = sj + q from the two vectors.  MODE 1: same, and mid is stored to `midbuf` (the first pass, when
// the output vector aliases no input and can serve as scratch).  MODE 2: `sj` IS the stored mid, q is not read:
// every later pass of the search moves 2R instead of 3R.
// GRAD (the solver step, MODE 0 and 1): the q plane holds ∇f, and q = mnu ∇f (mnu = -ν) is rounded to R before the
// sum, as the caller's broadcast rounds it (-fmad=false keeps the product out of an FMA): mid, and so every sum of
// the pass, is bit for bit the prox!'s of that q.
template <class R, int K, int VEC, int MODE, bool GRAD>
__global__ void __launch_bounds__(kEwThreads, L1b2Unroll<R, K>::minb)
    l1b2_norm_kernel(const R* xk, const R* sj, const R* q, R* midbuf, long long n, R ls, bool use_scale,
                     ScaleSet<K> sc, int nblocks_stride, Partial* __restrict__ partials, R mnu) {
  static_assert(!(GRAD && MODE == 2), "MODE 2 does not read q");
  double acc[K], dot[K];
#pragma unroll
  for (int k = 0; k < K; ++k) { acc[k] = 0.0; dot[k] = 0.0; }
  double poison = 0.0;
  R scale[K];
#pragma unroll
  for (int k = 0; k < K; ++k) scale[k] = (R)sc.s[k];
  const long long nvec = n / VEC;
  // one packet of VEC elements: products summed in R over the packet (4 terms for Float32: conversions to
  // Float64 are quarter-rate, one per packet and trial instead of two per element), then added in Float64
  auto packet = [&](const R* x, const R* s, const R* qq, int m, R* mid_out) {
    R lo[VEC], hi[VEC], nx[VEC];
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
      const bool on = e < m;
      const R mid = on ? (MODE == 2 ? s[e] : s[e] + (GRAD ? mnu * qq[e] : qq[e])) : R(0);
      if (MODE == 1) mid_out[e] = mid;
      lo[e] = mid - ls;
      hi[e] = mid + ls;
      nx[e] = on ? -x[e] : R(0);
      poison += (double)(mid - mid);
      if (sizeof(R) == 4 && nx[e] != nx[e]) poison = (double)nx[e];  // a NaN in xk makes every norm NaN (see below)
      if (!on) { lo[e] = R(0); hi[e] = R(0); }
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
      if (sizeof(R) == 8) {
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
          const R z = use_scale ? nx[e] * scale[k] : nx[e];
          const bool below = z < lo[e], above = z > hi[e];
          const R w = below ? lo[e] : (above ? hi[e] : z);
          const R dw = (below || above) ? R(0) : nx[e];
          acc[k] = __fma_rn((double)w, (double)w, acc[k]);
          dot[k] = __fma_rn((double)w, (double)dw, dot[k]);
        }
      } else {
        // Float32: the clamp as two FMNMX and the derivative term as one predicated FMA (w == z exactly when z is not
        // clamped): 6 instructions per element and trial instead of 9 -- the 2R passes are issue-bound in Float32
        // (1.26 ms at 2^29 against 0.66 ms of HBM time).  Same values in the same order as the compare-and-select
        // form; FMNMX drops a NaN z, which the xk-NaN flag of the packet (below) puts back.
        float pa = 0.0f, pd = 0.0f;
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
          const float z = use_scale ? (float)nx[e] * (float)scale[k] : (float)nx[e];
          const float w = fminf(fmaxf(z, (float)lo[e]), (float)hi[e]);
          pa = fmaf(w, w, pa);
          pd = (w == z) ? fmaf(w, (float)nx[e], pd) : pd;
        }
        acc[k] += (double)pa;
        dot[k] += (double)pd;
      }
    }
  };
  // U packets per thread and trip, all loads issued before the first use: a 2R pass keeps only 32 B per
  // thread in flight otherwise, too little to cover the HBM latency at the occupancy the K accumulators allow
  constexpr int U = L1b2Unroll<R, K>::value;
  for (long long v0 = (long long)blockIdx.x * (kEwThreads * U) + threadIdx.x; v0 < nvec;
       v0 += (long long)gridDim.x * (kEwThreads * U)) {
    Pack<R, VEC> a[U], b[U], c[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long v = v0 + (long long)u * kEwThreads;
      if (v < nvec) {
        ld_stream(xk + v * VEC, a[u]);
        ld_stream(sj + v * VEC, b[u]);
        if (MODE != 2) ld_stream(q + v * VEC, c[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long v = v0 + (long long)u * kEwThreads;
      if (v < nvec) {
        Pack<R, VEC> mo;
        packet(a[u].v, b[u].v, c[u].v, VEC, mo.v);
        if (MODE == 1) st_stream(midbuf + v * VEC, mo);
      }
    }
  }
  if (VEC > 1 && blockIdx.x == gridDim.x - 1) {
    const long long i = nvec * VEC + threadIdx.x;
    if (i < n) {
      R x1[VEC] = {xk[i]}, s1[VEC] = {sj[i]}, q1[VEC] = {MODE != 2 ? q[i] : R(0)}, m1[VEC];
      packet(x1, s1, q1, 1, m1);
      if (MODE == 1) midbuf[i] = m1[0];
    }
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
    Partial p;
    p.s = dot[k];
    p.s2 = acc[k] + poison;
    p.bad = -1;
    p = block_fold<kEwThreads>(p);
    if (threadIdx.x == 0) partials[(size_t)k * nblocks_stride + blockIdx.x] = p;
  }
}

template <class R, int K>
static int32_t norm_pass_k(spx_ctx* ctx, int64_t n, const R* xk, const R* sj, const R* q, R ls, const double* scale,
                           int nscale, double* out, double* dot_out, int mode, R* midbuf, bool grad, R mnu) {
  ScaleSet<K> sc;
  for (int k = 0; k < K; ++k) sc.s[k] = scale ? scale[k < nscale ? k : nscale - 1] : 1.0;
  const uintptr_t bits = (uintptr_t)xk | (uintptr_t)sj | (uintptr_t)q | (uintptr_t)midbuf;
  const bool vec = (bits & 15u) == 0;
  constexpr int VECW = 16 / (int)sizeof(R);
  const long long nv = vec ? n / VECW : n;
  long long want = (nv + kEwThreads * L1b2Unroll<R, K>::value - 1) / (kEwThreads * L1b2Unroll<R, K>::value);
  if (want < 1) want = 1;
  long long cap = (long long)ctx->sm_count * 8;
  const int grid = (int)(want < cap ? want : cap);
#define SPX_L1B2_LAUNCH(V, M, G)                                                                                \
  l1b2_norm_kernel<R, K, V, M, G><<<grid, kEwThreads, 0, ctx->stream>>>(xk, sj, q, midbuf, n, ls, scale != nullptr, \
                                                                        sc, grid, ctx->d_partials, mnu)
#define SPX_L1B2_MODES(V)                                                  \
  if (mode == 2) SPX_L1B2_LAUNCH(V, 2, false);                             \
  else if (mode == 1 && grad) SPX_L1B2_LAUNCH(V, 1, true);                 \
  else if (mode == 1) SPX_L1B2_LAUNCH(V, 1, false);                        \
  else if (grad) SPX_L1B2_LAUNCH(V, 0, true);                              \
  else SPX_L1B2_LAUNCH(V, 0, false)
  if (vec) {
    SPX_L1B2_MODES(VECW);
  } else {
    SPX_L1B2_MODES(1);
  }
#undef SPX_L1B2_MODES
#undef SPX_L1B2_LAUNCH
  ctx->launches++;
  SPX_CUDA(cudaGetLastError());
  int32_t st = finalize_partials(ctx, grid, K, false);
  if (st != SPX_OK) return st;
  for (int k = 0; k < nscale; ++k) out[k] = ctx->h_result[k].s2;
  if (dot_out)
    for (int k = 0; k < nscale; ++k) dot_out[k] = ctx->h_result[k].s;
  return SPX_OK;
}

template <class R>
static int32_t norm_pass(spx_ctx* ctx, int64_t n, const R* xk, const R* sj, const R* q, R ls, const double* scale,
                         int nscale, double* out, double* dot_out = nullptr, int mode = 0, R* midbuf = nullptr,
                         bool grad = false, R mnu = R(0)) {
  if (n == 0) {
    for (int k = 0; k < nscale; ++k) out[k] = 0.0;
    if (dot_out)
      for (int k = 0; k < nscale; ++k) dot_out[k] = 0.0;
    return SPX_OK;
  }
  if (nscale <= 1) return norm_pass_k<R, 1>(ctx, n, xk, sj, q, ls, scale, nscale, out, dot_out, mode, midbuf, grad, mnu);
  if (nscale <= 4) return norm_pass_k<R, 4>(ctx, n, xk, sj, q, ls, scale, nscale, out, dot_out, mode, midbuf, grad, mnu);
  if (nscale <= 8) return norm_pass_k<R, 8>(ctx, n, xk, sj, q, ls, scale, nscale, out, dot_out, mode, midbuf, grad, mnu);
  return norm_pass_k<R, 16>(ctx, n, xk, sj, q, ls, scale, nscale, out, dot_out, mode, midbuf, grad, mnu);
}

// y = ProjB(-xk scale) post - sj (L1B2Finish, spx_ops.cuh), with Σ|xk+sj+y| and Σ(sj+y)² for ψ(y)
template <class R>
static int32_t finish_pass(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q, R ls, bool use_scale,
                           R scale, R post, double* psi_sum, double* w_sumsq, bool have_mid = false) {
  const bool psi = psi_sum != nullptr || w_sumsq != nullptr;
  int nb = 0;
  int32_t st;
  if (psi) {
    L1B2Finish<R, true> op;
    op.in[0] = xk; op.in[1] = sj; op.in[2] = q;
    op.fill[0] = op.fill[1] = op.fill[2] = R(0);
    op.y = y; op.ls = ls; op.scale = scale; op.post = post; op.use_scale = use_scale;
    op.have_mid = have_mid;
    if (have_mid) op.in[2] = y;
    st = ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, &nb);
    if (st != SPX_OK) return st;
    st = finalize_partials(ctx, nb, 1, false);
    if (st != SPX_OK) return st;
    if (psi_sum) *psi_sum = ctx->h_result[0].s;
    if (w_sumsq) *w_sumsq = ctx->h_result[0].s2;
    return SPX_OK;
  }
  L1B2Finish<R, false> op;
  op.in[0] = xk; op.in[1] = sj; op.in[2] = q;
  op.fill[0] = op.fill[1] = op.fill[2] = R(0);
  op.y = y; op.ls = ls; op.scale = scale; op.post = post; op.use_scale = use_scale;
  op.have_mid = have_mid;
  if (have_mid) op.in[2] = y;
  return ew_launch(ctx, ctx->stream, op, n, 0, ctx->d_partials, &nb);
}

template <class R> static bool in_ball_l2(R nw, R delta) {
  const R eps = std::numeric_limits<R>::epsilon();
  if (nw <= delta) return true;
  if (!std::isfinite(nw) || !std::isfinite(delta)) return false;
  R tol = std::max(eps, std::sqrt(eps) * std::max(std::fabs(nw), std::fabs(delta)));
  return std::fabs(nw - delta) <= tol;
}

// What the search reads and writes.  prox!: q is the q vector; the finish writes y and sums ψ's two sums.  The solver
// step (spx_step_l1b2): the q plane holds ∇f and every pass forms q = fl(mnu ∇f), mnu = -ν, on the load, so every sum of
// the search is the prox!'s of that q bit for bit; the finish also writes xsy (may be NULL) and sums Σs², Σ∇f·s.
template <class R> struct L1B2Io {
  R* y;
  const R *xk, *sj, *q;
  bool grad = false;
  R mnu = R(0);
  R* xsy = nullptr;
  double* sums = nullptr;  // step: {Σs², Σ∇f·s}
};

template <class R>
static int32_t l1b2_search(spx_ctx* ctx, int64_t n, const L1B2Io<R>& io, double lambda_, double sigma_, double delta_,
                           double chi_lambda_, spx_allreduce_sum_fn reduce, void* user, int32_t* passes_out,
                           double* psi_out) {
  SPX_REQUIRE(ctx != nullptr, "null context");
  SPX_REQUIRE(n >= 0, "n < 0");
  R* const y = io.y;
  const R *const xk = io.xk, *const sj = io.sj, *const q = io.q;
  SPX_REQUIRE(n == 0 || (y && xk && sj && q), "null device vector");
  DeviceGuard guard(ctx->device);
  const R lam = (R)lambda_, sig = (R)sigma_, delta = (R)delta_, chil = (R)chi_lambda_;
  const R ls = lam * sig;
  const char* const who = io.grad ? "spx_step_l1b2" : "spx_prox_l1b2";  // the entry point, for error messages
  int passes = 0;
  // y as scratch for mid = sj + q while the search runs (2R per pass instead of 3R), and the finish as the check of an
  // unverified root (after a failed check the search re-reads its inputs): only when no output overlaps an input.
  // Otherwise (prox!(y, ψ, y, σ), or the step's x <- x + s) every pass reads xk, sj, q and the search converges by
  // evaluation; the finish reads each element's operands before it writes its outputs.
  auto clear_of_inputs = [&](const R* p) {
    const size_t bytes = (size_t)n * sizeof(R);
    return !spans_overlap(p, xk, bytes) && !spans_overlap(p, sj, bytes) && !spans_overlap(p, q, bytes);
  };
  const bool can_stash = n > 0 && clear_of_inputs(y) && clear_of_inputs(io.xsy);
  bool stashed = false;
  // K residuals per pass: f_k = η_k - χ(ProjB(-xk η_k/Δ)) and their derivatives
  // f'_k = 1 - χ (Σ w dw/dscale) / (‖w‖ Δ)
  auto eval = [&](const std::vector<R>& etas, bool use_scale, std::vector<R>& f, std::vector<R>& df) -> int32_t {
    const int m = (int)etas.size();
    double scale[kMaxScale], ss[2 * kMaxScale];
    for (int k = 0; k < m; ++k) scale[k] = (double)(etas[k] / delta);
    // the first pass decides whether the ball is active at all and leaves y alone; the second (the first of
    // the search proper) also stores mid into y; later passes read it back instead of sj and q
    const int mode = (!can_stash || passes == 0) ? 0 : (stashed ? 2 : 1);
    int32_t st = norm_pass<R>(ctx, n, xk, mode == 2 ? (const R*)y : sj, q, ls, use_scale ? scale : nullptr, m, ss,
                              ss + m, mode, y, io.grad && mode != 2, io.mnu);
    if (mode == 1) stashed = true;
    if (st != SPX_OK) return st;
    ++passes;
    if (reduce) {
      st = reduce(user, ss, 2 * m);
      if (st != SPX_OK) {
        set_error("%s: all-reduce callback failed (%d)", who, (int)st);
        return st;
      }
    }
    f.resize(m);
    df.resize(m);
    for (int k = 0; k < m; ++k) {
      const double nw = std::sqrt(ss[k]);
      f[k] = etas[k] - chil * (R)nw;
      df[k] = (R)(1.0 - (double)chil * ss[m + k] / (nw * (double)delta));
    }
    return SPX_OK;
  };
  // the finish pass: y = ProjB(-xk scale) post - sj and, when v is given, v = {Σ|xk+sj+y|, Σ(sj+y)²} -- for the step
  // always, with xsy written and v[2..3] = {Σs², Σ∇f·s} -- all-reduced in one call when the vector is sharded
  auto finish_pass_io = [&](bool use_scale, R scale, R post, double* v) -> int32_t {
    int32_t st = io.grad ? step_l1b2_finish<R>(ctx, n, y, io.xsy, xk, sj, q, stashed ? y : nullptr, sig, ls, use_scale,
                                               scale, post, v)
                         : finish_pass<R>(ctx, n, y, xk, sj, q, ls, use_scale, scale, post, v ? &v[0] : nullptr,
                                          v ? &v[1] : nullptr, stashed);
    ++passes;
    if (st != SPX_OK || v == nullptr || reduce == nullptr) return st;
    return reduce(user, v, io.grad ? 4 : 2);
  };
  // ψ(y) = h(xk+sj+y) + IndBallL2(Δ)(sj+y)   shiftedNormL1B2.jl:32;  the step's sums beside it
  auto results = [&](const double* v) {
    if (psi_out)
      *psi_out = in_ball_l2<R>((R)std::sqrt(v[1]), delta) ? (double)(lam * (R)v[0]) : std::numeric_limits<double>::infinity();
    if (io.sums) {
      io.sums[0] = v[2];
      io.sums[1] = v[3];
    }
  };
  auto finish = [&](bool use_scale, R scale, R post) -> int32_t {
    double v[4] = {0.0, 0.0, 0.0, 0.0};
    const bool sums = psi_out != nullptr || io.grad;
    int32_t st = finish_pass_io(use_scale, scale, post, sums ? v : nullptr);
    if (passes_out) *passes_out = passes;
    if (st != SPX_OK || !sums) return st;
    results(v);
    return SPX_OK;
  };

  // ---- the search -----------------------------------------------------------------------------------------------
  // The residual f(η) = η - χ(ProjB(-xk η/Δ)) is C¹ and increasing; every pass returns f and f' at up to four trial
  // values.  Pass 0 is a ladder Δ·{1, 2, 4, 16}: f(Δ) decides whether the ball is active (:58), the ladder brackets
  // the root.  Every further pass evaluates a cluster around the root x̂ of the cubic Hermite interpolant of f on the
  // current bracket, x̂ - e, x̂, x̂ + e and one point 3e out on the wider side, e = 2^-6 of the bracket for the first
  // cluster and 2^-16 afterwards (what the interpolant's error leaves: for large n, A(η) and B(η) of
  // ||·||² = (η/Δ)² A + B are smooth up to the granularity of single entries changing side).  The search ends on an
  // evaluated point with |f| <= 4 ulp(η), on an exact zero, or on two adjacent floats around the sign change (Roots'
  // end state); when the bracket is already narrower than the interpolant is accurate to an ulp, the FINISH pass takes
  // x̂ unevaluated and doubles as its check -- it returns Σ(sj + y)² = (||w|| Δ/η)², i.e. the residual at x̂ -- which
  // saves one pass over the vector; a failed check (never observed) re-enters the search.
  struct Pt { R x, f, d; };
  std::vector<Pt> known;
  std::vector<R> f, df, pts;
  for (double m : {1.0, 2.0, 4.0, 16.0}) {
    const R x = delta * (R)m;
    if (std::isfinite(x) && (pts.empty() || x > pts.back())) pts.push_back(x);
  }
  int32_t st = eval(pts, true, f, df);  // η = Δ: scale 1, i.e. ||ProjB(-xk)|| itself (:56-58)
  if (st != SPX_OK) return st;
  // f[0] = Δ - χ(y); the reference tests Δ <= χ(y)  (:58) -- the sign of a difference is exact
  if (!(f[0] <= R(0))) return finish(false, R(1), R(1));
  for (size_t k = 0; k < pts.size(); ++k) known.push_back({pts[k], f[k], df[k]});
  auto ulp_of = [](R x) -> R { return std::nextafter(x, std::numeric_limits<R>::infinity()) - x; };
  auto hermite_root = [](R a, R fa, R da, R b, R fb, R db) -> R {  // root of the cubic Hermite interpolant in (a, b)
    const double h = (double)b - (double)a;
    auto p = [&](double x) {
      const double t = (x - (double)a) / h, t2 = t * t, t3 = t2 * t;
      return (2 * t3 - 3 * t2 + 1) * (double)fa + (t3 - 2 * t2 + t) * h * (double)da + (-2 * t3 + 3 * t2) * (double)fb +
             (t3 - t2) * h * (double)db;
    };
    double lo = (double)a, hi = (double)b;
    for (int it = 0; it < 200; ++it) {
      const double mid = 0.5 * (lo + hi);
      if (!(lo < mid && mid < hi)) break;
      if ((p(mid) < 0.0) == ((double)fa < 0.0)) lo = mid;
      else hi = mid;
    }
    return (R)(0.5 * (lo + hi));
  };
  R eta = delta;
  int clusters = 0;
  bool unverified_ok = can_stash;  // a failed check re-reads the inputs, which y (and xsy) must not have overwritten
  R b0 = std::max(R(2) * pts.back(), pts.back() + R(1));
  for (;;) {
    // bracket = the largest evaluated point with f < 0 and the smallest with f > 0 (f is increasing)
    const Pt *pa = nullptr, *pb = nullptr, *pz = nullptr, *best = &known[0];
    for (const Pt& k : known) {
      if (k.f == R(0)) pz = &k;
      if (k.f < R(0) && (!pa || k.x > pa->x)) pa = &k;
      if (k.f > R(0) && (!pb || k.x < pb->x)) pb = &k;
      if (std::fabs(k.f) < std::fabs(best->f)) best = &k;
    }
    if (pz) { eta = pz->x; break; }
    if (!pa || passes > 200) {
      set_error("%s: no sign change of the trust-region residual", who);
      return SPX_E_NOROOT;
    }
    if (!pb) {  // the ladder did not reach the root: the reference's own guesses max(2a, a+1) 4^k, and a Newton point
      pts.clear();
      const R xn = (pa->d > R(0)) ? pa->x - pa->f / pa->d : std::numeric_limits<R>::infinity();
      if (std::isfinite(xn) && xn > pa->x) {
        pts.push_back(xn);
        pts.push_back(xn + (xn - pa->x));
      }
      for (int k = 0; k < 2; ++k) pts.push_back(b0 * (R)std::ldexp(1.0, 2 * k));
      b0 = b0 * R(16);
      std::sort(pts.begin(), pts.end());
      pts.erase(std::unique(pts.begin(), pts.end()), pts.end());
      while (!pts.empty() && !(std::isfinite(pts.back()) && pts.back() > pa->x)) pts.pop_back();
      std::vector<R> in;
      for (R x : pts)
        if (x > pa->x) in.push_back(x);
      if (in.empty()) {
        set_error("%s: no sign change of the trust-region residual", who);
        return SPX_E_NOROOT;
      }
      st = eval(in, true, f, df);
      if (st != SPX_OK) return st;
      for (size_t k = 0; k < in.size(); ++k) known.push_back({in[k], f[k], df[k]});
      continue;
    }
    const R a = pa->x, b = pb->x;
    if (std::fabs(best->f) <= R(4) * ulp_of(best->x)) { eta = best->x; break; }
    const R mid = a + (b - a) / R(2);
    if (!(a < mid && mid < b)) {  // adjacent floats around the sign change
      eta = (std::fabs(pa->f) <= std::fabs(pb->f)) ? a : b;
      break;
    }
    R xh = hermite_root(a, pa->f, pa->d, b, pb->f, pb->d);
    if (!(xh > a && xh < b)) xh = mid;
    const R width = b - a;
    // bracket narrow enough for the interpolant to be good to an ulp: x̂ goes to the finish pass, which checks it
    const R narrow = (sizeof(R) == 8 ? R(1e-6) : R(2e-4)) * a;
    if (unverified_ok && clusters >= 1 && width <= narrow) {
      double v[4] = {0.0, 0.0, 0.0, 0.0};
      const R scale = xh / delta, post = delta / xh;
      st = finish_pass_io(true, scale, post, v);
      if (st != SPX_OK) return st;
      stashed = false;  // y now holds the result, not sj + q
      // ||w|| = ||sj + y|| η/Δ;  f(x̂) = x̂ - χ ||w||
      const R nw = (R)(std::sqrt(v[1]) * ((double)xh / (double)delta));
      const R fx = xh - chil * nw;
      if (std::fabs(fx) <= R(8) * ulp_of(xh)) {
        if (passes_out) *passes_out = passes;
        results(v);
        return SPX_OK;
      }
      unverified_ok = false;  // re-enter the search with what the check measured (slope unknown: reuse the nearer end's)
      known.push_back({xh, fx, (xh - a < b - xh) ? pa->d : pb->d});
      continue;
    }
    const int kbits = clusters == 0 ? 6 : 16;
    R e = std::max(R(4) * ulp_of(xh), width * (R)std::ldexp(1.0, -kbits));
    const R far = (b - xh > xh - a) ? xh + R(3) * e : xh - R(3) * e;
    const R cand[4] = {xh - e, xh, xh + e, far};
    pts.assign(cand, cand + 4);
    std::sort(pts.begin(), pts.end());
    std::vector<R> in;
    for (R x : pts)
      if (x > a && x < b && (in.empty() || x > in.back())) in.push_back(x);
    if (in.empty()) in.push_back(mid);
    st = eval(in, true, f, df);
    if (st != SPX_OK) return st;
    for (size_t k = 0; k < in.size(); ++k) known.push_back({in[k], f[k], df[k]});
    ++clusters;
  }
  return finish(true, eta / delta, delta / eta);
}

template <class R>
static int32_t prox_l1b2(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q, double lambda,
                         double sigma, double delta, double chi_lambda, spx_allreduce_sum_fn reduce, void* user,
                         int32_t* passes_out, double* psi_out) {
  L1B2Io<R> io;
  io.y = y; io.xk = xk; io.sj = sj; io.q = q;
  return l1b2_search<R>(ctx, n, io, lambda, sigma, delta, chi_lambda, reduce, user, passes_out, psi_out);
}

// the solver step: the search with σ = ν on q = fl(-ν∇f), formed from ∇f inside its passes
template <class R>
static int32_t step_l1b2(spx_ctx* ctx, int64_t n, R* s, R* xsy, const R* xk, const R* sj, const R* grad, double lambda,
                         double nu, double delta, double chi_lambda, spx_allreduce_sum_fn reduce, void* user,
                         int32_t* passes_out, double* out3) {
  SPX_STEP_COMMON_CHECKS("spx_step_l1b2", STEP_L1B2, n, out3);
  L1B2Io<R> io;
  io.y = s; io.xk = xk; io.sj = sj; io.q = grad;
  io.grad = true;
  io.mnu = -(R)nu;
  io.xsy = xsy;
  io.sums = out3 + 1;
  return l1b2_search<R>(ctx, n, io, lambda, nu, delta, chi_lambda, reduce, user, passes_out, out3);
}

}  // namespace spx

using namespace spx;

#define SPX_DEFINE_L1B2(SUF, R)                                                                                     \
  extern "C" int32_t spx_prox_l1b2_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q,       \
                                         double lambda, double sigma, double delta, double chi_lambda,              \
                                         int32_t* passes_out, double* psi_out) {                                    \
    return prox_l1b2<R>(ctx, n, y, xk, sj, q, lambda, sigma, delta, chi_lambda, nullptr, nullptr, passes_out,       \
                        psi_out);                                                                                   \
  }                                                                                                                 \
  extern "C" int32_t spx_prox_l1b2_sharded_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj,           \
                                                 const R* q, double lambda, double sigma, double delta,             \
                                                 double chi_lambda, spx_allreduce_sum_fn reduce, void* user,        \
                                                 int32_t* passes_out, double* psi_out) {                            \
    return prox_l1b2<R>(ctx, n, y, xk, sj, q, lambda, sigma, delta, chi_lambda, reduce, user, passes_out, psi_out); \
  }                                                                                                                 \
  extern "C" int32_t spx_step_l1b2_##SUF(spx_ctx* ctx, int64_t n, R* s, R* xsy, const R* xk, const R* sj,           \
                                         const R* grad, double lambda, double nu, double delta, double chi_lambda,  \
                                         int32_t* passes_out, double* out3) {                                       \
    return step_l1b2<R>(ctx, n, s, xsy, xk, sj, grad, lambda, nu, delta, chi_lambda, nullptr, nullptr, passes_out,  \
                        out3);                                                                                      \
  }                                                                                                                 \
  extern "C" int32_t spx_step_l1b2_sharded_##SUF(spx_ctx* ctx, int64_t n, R* s, R* xsy, const R* xk, const R* sj,   \
                                                 const R* grad, double lambda, double nu, double delta,             \
                                                 double chi_lambda, spx_allreduce_sum_fn reduce, void* user,        \
                                                 int32_t* passes_out, double* out3) {                               \
    return step_l1b2<R>(ctx, n, s, xsy, xk, sj, grad, lambda, nu, delta, chi_lambda, reduce, user, passes_out,      \
                        out3);                                                                                      \
  }                                                                                                                 \
  extern "C" int32_t spx_l1b2_projnorm2_##SUF(spx_ctx* ctx, int64_t n, const R* xk, const R* sj, const R* q,        \
                                              double lambda, double sigma, int32_t nscale,                          \
                                              const double* scale_host, double* sumsq_out_host) {                   \
    SPX_REQUIRE(ctx && sumsq_out_host, "null argument");                                                            \
    SPX_REQUIRE(n >= 0 && nscale >= 1 && nscale <= kMaxScale, "bad sizes");                                         \
    SPX_REQUIRE(n == 0 || (xk && sj && q), "null device vector");                                                   \
    DeviceGuard g(ctx->device);                                                                                     \
    return norm_pass<R>(ctx, n, xk, sj, q, (R)lambda * (R)sigma, scale_host, scale_host ? nscale : 1,               \
                        sumsq_out_host);                                                                            \
  }                                                                                                                 \
  extern "C" int32_t spx_l1b2_finish_##SUF(spx_ctx* ctx, int64_t n, R* y, const R* xk, const R* sj, const R* q,     \
                                           double lambda, double sigma, int32_t use_scale, double scale,            \
                                           double post, double delta, double* psi_sum_out, double* w_sumsq_out) {   \
    SPX_REQUIRE(ctx != nullptr, "null context");                                                                    \
    SPX_REQUIRE(n >= 0, "n < 0");                                                                                   \
    SPX_REQUIRE(n == 0 || (y && xk && sj && q), "null device vector");                                              \
    (void)delta;                                                                                                    \
    DeviceGuard g(ctx->device);                                                                                     \
    return finish_pass<R>(ctx, n, y, xk, sj, q, (R)lambda * (R)sigma, use_scale != 0, (R)scale, (R)post,            \
                          psi_sum_out, w_sumsq_out);                                                                \
  }

SPX_DEFINE_L1B2(f64, double)
SPX_DEFINE_L1B2(f32, float)
