// spx_setup.cuh -- host-side configuration of the prox! functors of spx_ops.cuh (operand slots and the
// loop-invariant scalars the reference computes ahead of its loops), shared by the entry points of
// spx_elementwise.cu and the fused solver step of spx_step.cu.
#pragma once
#include "spx_ops.cuh"

namespace spx {

static const double kInf = std::numeric_limits<double>::infinity();

template <class Op, class R> static inline void set3(Op& op, const R* a, const R* b, const R* c) {
  op.in[0] = a; op.in[1] = b; op.in[2] = c;
  for (int k = 0; k < Op::NIN; ++k) op.fill[k] = R(0);
}

// inputs of the Box functors: 0 xk, 1 sj, 2 q (or g), [3 d], then l, u (NULL -> the scalar)
template <class Op, class R>
static inline void set_box(Op& op, const R* xk, const R* sj, const R* qg, const R* d, const R* lvec, R lval,
                           const R* uvec, R uval) {
  int k = 0;
  op.in[k] = xk; op.fill[k++] = R(0);
  op.in[k] = sj; op.fill[k++] = R(0);
  op.in[k] = qg; op.fill[k++] = R(0);
  if (Op::NIN == 6) { op.in[k] = d; op.fill[k++] = R(0); }
  op.in[k] = lvec; op.fill[k++] = lval;
  op.in[k] = uvec; op.fill[k++] = uval;
}

// operands and λ of the iprox! functors, shared by iprox! (spx_elementwise.cu) and the fused istep (spx_step.cu).
// Unboxed (IproxL1 / IproxL0): xk, sj, g, d (d's fill is never read: d must be a vector)
template <class Op, class R>
static inline void set_iprox(Op& op, R* y, const R* xk, const R* sj, const R* g, const R* d, R lambda) {
  set3(op, xk, sj, g);
  op.in[3] = d;
  op.fill[3] = R(1);
  op.y = y;
  op.lambda = lambda;
}
// Box (IproxL1Box / IproxL0Box): set_box, the selection, λ and lam_ok -- λ is 0 or a normal number far enough from
// the range limits for the one-reciprocal quotients (quot4 / quot3 in spx_ops.cuh)
static inline bool lam_within(double lambda, double lo, double hi) {
  return lambda == 0.0 || (std::fabs(lambda) > lo && std::fabs(lambda) < hi);
}
template <class R, bool PSI> static inline void set_lam_ok(IproxL1Box<R, PSI>& op) {
  op.lam_ok = lam_within((double)op.lambda, 1e-100, 1e100);
}
template <class R, bool PSI> static inline void set_lam_ok(IproxL0Box<R, PSI>& op) {
  op.lam_ok = lam_within((double)op.lambda, 1e-150, 1e150);
}
template <class Op, class R>
static inline void set_iprox_box(Op& op, R* y, const R* xk, const R* sj, const R* g, const R* d, const R* lvec, R lval,
                                 const R* uvec, R uval, DevSel sel, R lambda) {
  set_box(op, xk, sj, g, d, lvec, lval, uvec, uval);
  op.y = y;
  op.sel = sel;
  op.lambda = lambda;
  set_lam_ok(op);
}

// λ·Σ in R, returned as double (NormL1/NormL0/RootNormLhalf value functors)
template <class R> static inline double scale_value(int kind, R lambda, double sum, int64_t r) {
  if (kind == SPX_H_INDBALLL0) return sum <= (double)r ? 0.0 : kInf;
  return (double)(lambda * (R)sum);
}

// 54^(1/3) (2νλ)^(2/3) / 4 in Float64  (shiftedRootNormLhalf.jl:49)
template <class R> static inline double lhalf_threshold(R nulam) {
  return std::pow(54.0, 1.0 / 3.0) * std::pow((double)(R(2) * nulam), 2.0 / 3.0) / 4.0;
}

// loop-invariant scalars of each prox! (λ and σ already rounded to R)
template <class R, bool PSI> static inline void configure(ProxL1<R, PSI>& op, R lam, R sig) {
  op.a = lam * sig;  // λσ  shiftedNormL1.jl:46
}
template <class R, bool PSI> static inline void configure(ProxL0<R, PSI>& op, R lam, R sig) {
  op.c = std::sqrt(R(2) * lam * sig);  // sqrt(2λσ)  shiftedNormL0.jl:44
}
template <class R, bool PSI> static inline void configure(ProxLhalf<R, PSI>& op, R lam, R sig) {
  const R nulam = sig * lam;  // shiftedRootNormLhalf.jl:47
  op.p = lhalf_threshold(nulam);
  op.c4 = (double)(nulam / R(4));
  op.c4f = (float)op.c4;
  op.fast = lhalf_f32_range_host(op.c4);
}
template <class R, bool PSI> static inline void configure(ProxL1Box<R, PSI>& op, R lam, R sig) {
  op.sl = sig * lam;  // σλ  shiftedNormL1Box.jl:95
}
template <class R, bool PSI> static inline void configure(ProxL0Box<R, PSI>& op, R lam, R sig) {
  op.c = R(2) * lam * sig;  // 2λσ  shiftedNormL0Box.jl:95
}
template <class R, bool PSI> static inline void configure(ProxLhalfBox<R, PSI>& op, R lam, R sig) {
  op.k.lambda = lam;
  op.k.c4 = (double)(sig * lam / R(4));
  op.k.by3.set(R(3));
  op.k.by_sigma.set(sig);
  op.k.by_sigma64.set((double)sig);
  op.kf = (float)(0.5 / (double)sig);
  op.lamf = (float)lam;
  op.c4f = (float)op.k.c4;
  op.a2 = op.k.c4 + op.k.c4;
  op.a2f = (float)op.a2;
  op.fast = lhalf_f32_range_host(op.k.c4) && lhalf_f32_range_host((double)sig) && lhalf_f32_range_host((double)lam);
}

static inline int box_kind(int opc) { return opc == BOX_L1 ? SPX_H_L1 : (opc == BOX_L0 ? SPX_H_L0 : SPX_H_LHALF); }

}  // namespace spx
