"""The oracle's composition of the fused step around iprox! (shiftedprox.istep_, spx_istep_sep_* / spx_istep_box_*).

The step's caller -- an iteration of a diagonal quasi-Newton solver (R2DH, TRDH of RegularizedOptimization.jl) -- is not
part of the reference, so the step is DEFINED here as the composition of the oracle's own iprox! and ψ(y) with Float64
sums, as oracle.solver_step does for prox!.  Parity unpinned beyond iprox! and ψ(y)."""
import numpy as np

from oracle import oracle as orc


def solver_istep(op, xk, sj, grad, D, dshift, lam, l=None, u=None, selected=None):
    """d = D .+ σ (rounded to the vectors' type);  s = iprox!(ψ, ∇f, d);  xsy = xk .+ sj .+ s;  ψ(s);  ‖s‖₂;  ∇f's;  sᵀ d s

    op: "l1" | "l0"; with bounds (l, u) the Box form of the same h.  An unboxed form raises AssertionError on a
    d[i] <= 0, as its iprox! does.  Returns (s, xsy, ψ(s), ‖s‖₂, ∇f's, sᵀ d s) -- the three sums in Float64."""
    dt = grad.dtype
    d = (D + dt.type(dshift)).astype(dt)
    if l is None:
        s = {"l1": orc.iprox_l1, "l0": orc.iprox_l0}[op](xk, sj, grad, d, lam)
        psi = orc.value_plain(op, xk, sj, s, lam)
    else:
        s = orc.iprox_box(op, xk, sj, grad, d, l, u, lam, selected)
        psi = orc.value_box(op, xk, sj, s, l, u, lam, selected)
    xsy = ((xk + sj) + s).astype(dt)
    s64, g64, d64 = s.astype(np.float64), grad.astype(np.float64), d.astype(np.float64)
    return (s, xsy, psi, float(np.sqrt(np.sum(s64 * s64))), float(np.sum(g64 * s64)),
            float(np.sum(d64 * s64 * s64)))
