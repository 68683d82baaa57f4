"""GPU parity of the solver step of ShiftedIndBallL0 / ShiftedIndBallL0BInf (include/shiftedprox.h:
spx_step_indballl0_*).

The step is  q = -ν∇f;  s = prox!(ψ, q, ν);  xsy = (xk + sj) + s;  ψ(s);  ‖s‖₂;  ∇f's.  A batch the stream top-r kernel
takes (>= 2 problems per SM, n % 8 == 0, 4096 <= n <= 131072, 0 < r < n, aligned, no output overlapping an input, xsy
given) runs it in one pass of that kernel, followed by the radix kernel and the fixup kernel for the problems it flags
(four launches with the fold); every other call takes the composed form inside the library.  Bars, for every case:
`s` bit-identical to the stand-alone prox! of fl(-ν∇f) into a separate buffer (the stream form itself) and to the
base-class composition ShiftedProximableFunction.step_, `xsy` bit-identical to (xk + sj) + s, ψ(s) exactly the type's
own ψ(s), ‖s‖ and ∇f's against Float64 sums (the scalars_close bars of test_gpu_step.py, NaN / Inf matched), and a
second call returning the same scalars.
"""
import math

import numpy as np
import pytest
import torch

from gpu_util import DEV, N, T, inputs, sp

pytestmark = pytest.mark.gpu

DT = [np.float64, np.float32]
NU, DELTA = 0.3, 0.5
NPROB = 300  # >= 2 x 148 SMs
ONE_PASS_LAUNCHES = 4  # stream step kernel, radix kernel on the flagged problems, fixup kernel, fold


def _same(a, b):
    return (math.isnan(a) and math.isnan(b)) or a == b


def _close(got, ref, rel, mag=None):
    if not math.isfinite(ref):
        assert _same(got, ref), (got, ref)
    elif mag is None:
        assert got == pytest.approx(ref, rel=rel, abs=1e-300)
    else:
        assert abs(got - ref) <= rel * mag, (got, ref, mag)


def _psi(r, xk, sj, binf, twice, nprob=NPROB):
    h = sp.IndBallL0(r)
    if binf:
        psi = sp.shifted(h, T(xk), DELTA, sp.NormLinf(1.0), nprob=nprob)
    else:
        psi = sp.shifted(h, T(xk), nprob=nprob)
    return sp.shifted(psi, T(sj)) if twice else psi


def _check(psi, xk, sj, grad, dt, one_pass, tgrad=None, s=None, xsy="new"):
    """One step: the bars of the module docstring.  xk, sj: the host copies of ψ's shifts (sj zeros when shifted once).
    Returns the StepResult."""
    n = grad.size
    tgrad = T(grad) if tgrad is None else tgrad
    s = torch.empty(n, dtype=tgrad.dtype, device=DEV) if s is None else s
    if isinstance(xsy, str):
        xsy = torch.empty(n, dtype=tgrad.dtype, device=DEV)
    l0 = sp.launch_count()
    out, res = sp.step_(s, psi, tgrad, NU, xsy=xsy)
    launches = sp.launch_count() - l0
    assert out is s
    assert (launches == ONE_PASS_LAUNCHES) == one_pass, launches
    gs = N(s).copy()
    gxsy = N(xsy).copy() if xsy is not None else None
    # the stand-alone prox! of fl(-ν∇f) into a separate buffer
    q = (dt(-dt(NU)) * grad).astype(dt)
    y = torch.empty(n, dtype=tgrad.dtype, device=DEV)
    sp.prox_(y, psi, T(q), NU)
    assert np.array_equal(gs, N(y), equal_nan=True), np.flatnonzero(~((gs == N(y)) | (np.isnan(gs) & np.isnan(N(y)))))[:8]
    if gxsy is not None:
        assert np.array_equal(gxsy, ((xk + sj) + gs).astype(dt), equal_nan=True)
    # ψ(s) exactly; the two sums against Float64 sums
    assert _same(res.psi, psi(s))
    g64, s64 = grad.astype(np.float64), gs.astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        ref_snorm = float(np.sqrt(np.sum(s64 * s64)))
        ref_gdots = float(np.sum(g64 * s64))
        mag = float(np.sum(np.abs(g64 * s64))) + 1e-300
    _close(res.snorm, ref_snorm, 1e-12)
    _close(res.gdots, ref_gdots, 1e-12, mag)
    # the base-class composition (spx_step_pre, prox! in place, ψ(s), spx_step_post)
    s2 = torch.empty_like(s)
    xsy2 = torch.empty_like(s) if xsy is not None else None
    _, res2 = sp.ShiftedProximableFunction.step_(psi, s2, tgrad, NU, xsy=xsy2)
    assert np.array_equal(N(s2), gs, equal_nan=True)
    if xsy is not None:
        assert np.array_equal(N(xsy2), gxsy, equal_nan=True)
    assert _same(res2.psi, res.psi)
    _close(res2.snorm, res.snorm, 1e-12)
    _close(res2.gdots, res.gdots, 1e-12, mag)
    # a second call gives the same scalars
    _, res3 = sp.step_(s, psi, tgrad, NU, xsy=xsy)
    assert all(_same(a, b) for a, b in zip(tuple(res3), tuple(res))), (tuple(res3), tuple(res))
    return res


def _batch(dt, pn, twice, seed_base=0):
    n = NPROB * pn
    xk, sj, grad = inputs(n, dt, base=seed_base)
    if not twice:
        sj = np.zeros_like(xk)
    return xk, sj, grad


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("pn,r", [(4096, 100), (4096, 3000), (8192 + 64, 700), (65_536, 1024), (65_536, 1)])
@pytest.mark.parametrize("binf", [False, True])
@pytest.mark.parametrize("twice", [False, True])
def test_step_topr_batch_one_pass(dt, pn, r, binf, twice):
    xk, sj, grad = _batch(dt, pn, twice)
    psi = _psi(r, xk, sj, binf, twice)
    res = _check(psi, xk, sj, grad, dt, one_pass=True)
    if not binf:
        assert res.psi == math.inf  # every problem keeps r entries: NPROB r > r over the batch


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("binf", [False, True])
def test_step_topr_guess_wrong_both_ways(dt, binf):
    """Problems of alternating scale (x1 / x1000): the threshold of the previous problem, which pass 1 uses to write
    the kept form early, is far too low on every other problem and far too high on the next, so pass 2b rewrites
    entries in both directions."""
    pn, r = 8192, 500
    xk, sj, grad = _batch(dt, pn, True, seed_base=3)
    scale = np.repeat(np.where(np.arange(NPROB) % 2 == 1, 1000.0, 1.0), pn).astype(dt)
    xk, sj, grad = (xk * scale).astype(dt), (sj * scale).astype(dt), (grad * scale).astype(dt)
    _check(_psi(r, xk, sj, binf, True), xk, sj, grad, dt, one_pass=True)


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("pn", [4096, 8192 + 64])
@pytest.mark.parametrize("binf", [False, True])
def test_step_topr_exact_ties_at_threshold(dt, pn, binf):
    """xk = sj = 0 and |∇f| on 64 values in [1, 2): every 16-bit key value holds ~pn / 64 exactly equal entries, so the
    threshold value is resolved by the candidate ranking (lowest index first) and its rewrites run on every problem."""
    rng = np.random.default_rng(7)
    n = NPROB * pn
    grad = (rng.choice([-1.0, 1.0], n) * (64 + rng.integers(0, 64, n)) / 64).astype(dt)
    xk, sj = np.zeros(n, dt), np.zeros(n, dt)
    _check(_psi(333, xk, sj, binf, True), xk, sj, grad, dt, one_pass=True)


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("pn", [4096, 65_536])
@pytest.mark.parametrize("binf", [False, True])
def test_step_topr_hard_problems_in_the_batch(dt, pn, binf):
    """Problems the stream kernel flags (crowded threshold value, constant, all zero, NaN, Inf; modelled on
    test_indballl0_batch_stream_form) go through the radix kernel in place and the fixup kernel: their s, xsy and sums
    are right and the sums include them."""
    r = 100
    xk, sj, grad = _batch(dt, pn, True, seed_base=6)
    special = {3: "ties", 7: "const", 11: "zero", 13: "nan", 17: "inf", NPROB - 1: "ties"}
    for p, kind in special.items():
        s = slice(p * pn, (p + 1) * pn)
        if kind == "ties":
            xk[s] = 0; sj[s] = 0
            grad[s] = (np.round(grad[s] * 2) / 2).astype(dt)
        elif kind == "const":
            xk[s] = 0; sj[s] = 0; grad[s] = dt(1.25)
        elif kind == "zero":
            xk[s] = 0; sj[s] = 0; grad[s] = 0
        elif kind == "nan":
            grad[p * pn + 5] = np.nan; grad[p * pn + pn - 2] = np.nan
        elif kind == "inf":
            grad[p * pn + 9] = np.inf; grad[p * pn + 77] = -np.inf
    _check(_psi(r, xk, sj, binf, True), xk, sj, grad, dt, one_pass=True)


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("binf", [False, True])
def test_step_topr_psi_zero(dt, binf):
    """xk + sj and ∇f zero outside one problem: r entries of the batch are non-zero, so ψ(s) = 0."""
    pn, r = 4096, 64
    n = NPROB * pn
    xk, sj = np.zeros(n, dt), np.zeros(n, dt)
    _, _, grad = _batch(dt, pn, True, seed_base=9)
    keep = slice(5 * pn, 6 * pn)
    g = np.zeros(n, dt)
    g[keep] = grad[keep]
    res = _check(_psi(r, xk, sj, binf, True), xk, sj, g, dt, one_pass=True)
    assert res.psi == 0.0


@pytest.mark.parametrize("dt", DT)
def test_step_topr_binf_infeasible(dt):
    """BInf: sj = 0.9Δ on the one non-zero problem, so the kept entries of sj + s leave the ball of 1.1Δ while the count
    of non-zeros stays within r: ψ(s) = Inf from the ball alone."""
    pn, r = 4096, 64
    n = NPROB * pn
    xk, sj = np.zeros(n, dt), np.zeros(n, dt)
    _, _, grad = _batch(dt, pn, True, seed_base=12)
    keep = slice(5 * pn, 6 * pn)
    sj[keep] = dt(0.9 * DELTA)
    g = np.zeros(n, dt)
    g[keep] = grad[keep]
    res = _check(_psi(r, xk, sj, True, True), xk, sj, g, dt, one_pass=True)
    assert res.psi == math.inf


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("binf", [False, True])
@pytest.mark.parametrize("case", ["few_problems", "n_not_mult_8", "unaligned", "xsy_none"])
def test_step_topr_composed_routes(dt, binf, case):
    """Calls outside the stream form's conditions take the composed form and give the base-class step's bits."""
    nprob, pn, r = NPROB, 4096, 100
    if case == "few_problems":
        nprob = 8
    elif case == "n_not_mult_8":
        pn = 4100
    xk, sj, grad = inputs(nprob * pn, dt, base=15)
    if case == "unaligned":  # views one element into their buffers: 8 (Float64) / 4 (Float32) bytes off 16
        n = nprob * pn
        bufs = [torch.empty(n + 1, dtype=T(grad).dtype, device=DEV) for _ in range(5)]
        vx, vs, vg, vout, vxsy = [b[1:] for b in bufs]
        vx.copy_(T(xk)); vs.copy_(T(sj)); vg.copy_(T(grad))
        h = sp.IndBallL0(r)
        psi = sp.shifted(h, vx, DELTA, sp.NormLinf(1.0), nprob=nprob) if binf else sp.shifted(h, vx, nprob=nprob)
        psi = sp.shifted(psi, vs)
        _check(psi, xk, sj, grad, dt, one_pass=False, tgrad=vg, s=vout, xsy=vxsy)
        return
    psi = _psi(r, xk, sj, binf, True, nprob=nprob)
    _check(psi, xk, sj, grad, dt, one_pass=False, xsy=None if case == "xsy_none" else "new")


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("binf", [False, True])
def test_step_topr_xsy_aliasing_xk(dt, binf):
    """xsy may be ψ's own xk (x + s written over x): the composed form, the same bits as the base-class step."""
    pn, r = 4096, 100
    xk, sj, grad = _batch(dt, pn, True, seed_base=18)
    psi1, psi2 = _psi(r, xk, sj, binf, True), _psi(r, xk, sj, binf, True)
    s1, s2 = torch.empty(xk.size, dtype=T(grad).dtype, device=DEV), torch.empty(xk.size, dtype=T(grad).dtype, device=DEV)
    tg = T(grad)
    l0 = sp.launch_count()
    _, res1 = sp.step_(s1, psi1, tg, NU, xsy=psi1.xk)
    assert sp.launch_count() - l0 != ONE_PASS_LAUNCHES
    _, res2 = sp.ShiftedProximableFunction.step_(psi2, s2, tg, NU, xsy=psi2.xk)
    assert np.array_equal(N(s1), N(s2), equal_nan=True)
    assert np.array_equal(N(psi1.xk), N(psi2.xk), equal_nan=True)
    assert np.array_equal(N(psi1.xk), ((xk + sj) + N(s1)).astype(dt), equal_nan=True)
    assert _same(res1.psi, res2.psi)
    assert res1.snorm == pytest.approx(res2.snorm, rel=1e-12)


@pytest.mark.parametrize("binf", [False, True])
def test_step_topr_s_aliasing_grad_raises(binf):
    xk, sj, grad = _batch(np.float64, 4096, True)
    psi = _psi(100, xk, sj, binf, True)
    g = T(grad)
    with pytest.raises(ValueError):
        sp.step_(g, psi, g, NU, xsy=torch.empty_like(g))
