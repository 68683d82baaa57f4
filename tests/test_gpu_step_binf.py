"""GPU parity of the solver step of ShiftedGroupNormL2Binf (include/shiftedprox.h: spx_step_groupl2binf_*).

The step is  q = -ν∇f;  s = prox!(ψ, q, ν);  xsy = (xk + sj) + s;  ψ(s);  ‖s‖₂;  ∇f's.  A uniform layout (n == ngroups m,
m = 16 ... 256) runs it in the one pass of the uniform-layout kernels; everything else takes the composed form inside the
library.  Bars: `s` bit-identical to the stand-alone prox! of fl(-ν∇f), `xsy` bit-identical to (xk + sj) + s, ψ(s)
against the type's own ψ(s) and the oracle's value, ‖s‖ and ∇f's against Float64 sums (scalars_close of
test_gpu_step.py), and the same bits as the base-class composition ShiftedProximableFunction.step_.
"""
import numpy as np
import pytest
import torch

from gpu_util import DEV, N, T, inputs, orc, sp
from test_gpu_step import scalars_close

pytestmark = pytest.mark.gpu

DT = [np.float64, np.float32]
NU, DELTA = 0.3, 0.5


def _psi(lam_g, offs, xk, sj, delta=DELTA, twice=True):
    h = sp.GroupNormL2(T(lam_g), None, offsets=T(offs))
    psi = sp.shifted(h, T(xk), delta, sp.NormLinf(1.0))
    return sp.shifted(psi, T(sj)) if twice else psi


def _check(psi, xk, sj, grad, offs, lam_g, dt, delta=DELTA, tgrad=None, s=None, xsy=None):
    """One step: the bars of the module docstring.  Returns (s, xsy, result) as host arrays / StepResult."""
    n = grad.size
    tgrad = T(grad) if tgrad is None else tgrad
    s = torch.empty(n, dtype=tgrad.dtype, device=DEV) if s is None else s
    xsy = torch.empty_like(s) if xsy is None else xsy
    out, res = sp.step_(s, psi, tgrad, NU, xsy=xsy)
    assert out is s
    q = (dt(-dt(NU)) * grad).astype(dt)
    y = torch.empty(n, dtype=tgrad.dtype, device=DEV)
    sp.prox_(y, psi, T(q), NU)
    gs = N(s)
    assert np.array_equal(gs, N(y), equal_nan=True)
    assert np.array_equal(N(xsy), ((xk + sj) + gs).astype(dt), equal_nan=True)
    g64, s64 = grad.astype(np.float64), gs.astype(np.float64)
    ref_psi = orc.value_binf("groupl2", xk, sj, gs, delta, offs=offs, lam_g=lam_g)
    scalars_close(res, ref_psi, float(np.sqrt(np.sum(s64 * s64))), float(np.sum(g64 * s64)), grad, gs, dt)
    assert res.psi == pytest.approx(psi(s), rel=1e-12 if dt == np.float64 else 1e-6, abs=1e-300)
    # the base-class composition (spx_step_pre, prox! in place with ψ(s) from its value pass, spx_step_post)
    s2, xsy2 = torch.empty_like(s), torch.empty_like(s)
    _, res2 = sp.ShiftedProximableFunction.step_(psi, s2, tgrad, NU, xsy=xsy2)
    assert np.array_equal(N(s2), gs, equal_nan=True) and np.array_equal(N(xsy2), N(xsy), equal_nan=True)
    rel = 1e-12 if dt == np.float64 else 1e-6
    assert res2.psi == pytest.approx(res.psi, rel=rel, abs=1e-300)
    assert res2.snorm == pytest.approx(res.snorm, rel=1e-12)
    mag = float(np.sum(np.abs(g64 * s64))) + 1e-300
    assert abs(res2.gdots - res.gdots) <= 1e-12 * mag
    return gs, N(xsy), res


def _uniform(dt, m, ng, lam_scale=1.0):
    n = ng * m
    offs = np.arange(0, n + 1, m)
    xk, sj, grad = inputs(n, dt)
    lam_g = ((dt(0.5) + orc.uniform(ng, 12, dt)) * dt(lam_scale)).astype(dt)
    return xk, sj, grad, offs, lam_g


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("m", [16, 32, 64, 128, 256])
@pytest.mark.parametrize("twice", [False, True])
def test_step_binf_uniform_layouts(dt, m, twice):
    """ngroups = 1203 is not a multiple of 32/L for m < 256: the last round is partial."""
    xk, sj, grad, offs, lam_g = _uniform(dt, m, 1203)
    if not twice:
        sj = np.zeros_like(sj)
    psi = _psi(lam_g, offs, xk, sj, twice=twice)
    _, _, res = _check(psi, xk, sj, grad, offs, lam_g, dt)
    assert np.isfinite(res.psi)
    # xsy is optional, and a second identical call returns the same scalars
    s2 = torch.empty(grad.size, dtype=T(grad).dtype, device=DEV)
    _, res2 = sp.step_(s2, psi, T(grad), NU)
    assert tuple(res2) == tuple(res)


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("plant", ["huge", "nan", "big_lambda"])
def test_step_binf_declined_rounds(dt, plant):
    """Rounds the fast search declines go through the bracketing search of the second launch: magnitudes beyond its
    Float32 range guards, a NaN in ∇f, λ_g × 200.  s stays bit-identical to prox!, and two identical calls return
    identical scalars although the work list of declined rounds is filled in atomicAdd order."""
    m, ng = 64, 20_011
    xk, sj, grad, offs, lam_g = _uniform(dt, m, ng, 200.0 if plant == "big_lambda" else 1.0)
    if plant == "huge":  # |sol| ~ 1e13 .. 3e13 on every 97th group (Float32 squares of the search would overflow)
        for g in range(5, ng, 97):
            grad[g * m:(g + 1) * m] *= dt(1e13)
    elif plant == "nan":
        grad[777 * m + 5] = np.nan
    psi = _psi(lam_g, offs, xk, sj)
    if plant == "nan":
        s = torch.empty(grad.size, dtype=T(grad).dtype, device=DEV)
        xsy = torch.empty_like(s)
        _, res = sp.step_(s, psi, T(grad), NU, xsy=xsy)
        q = (dt(-dt(NU)) * grad).astype(dt)
        y = torch.empty_like(s)
        sp.prox_(y, psi, T(q), NU)
        assert np.array_equal(N(s), N(y), equal_nan=True)
        assert np.array_equal(N(xsy), ((xk + sj) + N(s)).astype(dt), equal_nan=True)
        ok = np.ones(grad.size, bool)
        ok[777 * m:778 * m] = False
        assert np.isfinite(N(s)[ok]).all()
        _, res2 = sp.step_(torch.empty_like(s), psi, T(grad), NU)
        assert np.array_equal(np.array(tuple(res2)), np.array(tuple(res)), equal_nan=True)
        return
    _, _, res = _check(psi, xk, sj, grad, offs, lam_g, dt)
    for _ in range(2):
        _, res2 = sp.step_(torch.empty(grad.size, dtype=T(grad).dtype, device=DEV), psi, T(grad), NU)
        assert tuple(res2) == tuple(res)


@pytest.mark.parametrize("dt", DT)
def test_step_binf_infeasible(dt):
    """A trust region far below the rounding of sj + s (Δ = 1e-20 / 1e-12): the composed ψ(s) is Inf, and so is the
    one-pass one."""
    delta = 1e-20 if dt == np.float64 else 1e-12
    xk, sj, grad, offs, lam_g = _uniform(dt, 64, 1203)
    psi = _psi(lam_g, offs, xk, sj, delta=delta)
    s2 = torch.empty(grad.size, dtype=T(grad).dtype, device=DEV)
    _, rc = sp.ShiftedProximableFunction.step_(psi, s2, T(grad), NU)
    assert rc.psi == np.inf
    _, _, res = _check(psi, xk, sj, grad, offs, lam_g, dt, delta=delta)
    assert res.psi == np.inf


@pytest.mark.parametrize("dt", DT)
def test_step_binf_fallbacks(dt):
    """Layouts and arguments the one-pass form does not take give the composed result: a ragged layout, unaligned views,
    ν outside the range of the fast searches, offsets rewritten in place so that the layout is no longer uniform (found
    on the device: the kernels raise the redo flag), n == 0 and a single group."""
    from test_gpu_parity import ragged_offsets

    # ragged
    offs = ragged_offsets(300, 256)
    n = int(offs[-1])
    xk, sj, grad = inputs(n, dt)
    lam_g = (dt(0.5) + orc.uniform(len(offs) - 1, 12, dt)).astype(dt)
    _check(_psi(lam_g, offs, xk, sj), xk, sj, grad, offs, lam_g, dt)
    # unaligned views: every vector one element into its allocation
    m, ng = 64, 1203
    xk, sj, grad, offs, lam_g = _uniform(dt, m, ng)
    n = ng * m
    pad = lambda a: T(np.concatenate([[0], a]).astype(dt))[1:]  # noqa: E731
    h = sp.GroupNormL2(T(lam_g), None, offsets=T(offs))
    psi_u = sp.shifted(sp.shifted(h, pad(xk), DELTA, sp.NormLinf(1.0)), pad(sj))
    s = torch.empty(n + 1, dtype=T(grad).dtype, device=DEV)[1:]
    xsy = torch.empty(n + 1, dtype=s.dtype, device=DEV)[1:]
    _check(psi_u, xk, sj, grad, offs, lam_g, dt, tgrad=pad(grad), s=s, xsy=xsy)
    # ν outside the range of the branch-free quotient
    psi = _psi(lam_g, offs, xk, sj)
    s = torch.empty(n, dtype=T(grad).dtype, device=DEV)
    _, r_small = sp.step_(s, psi, T(grad), 1e-31)
    s2 = torch.empty_like(s)
    _, r_small2 = sp.ShiftedProximableFunction.step_(psi, s2, T(grad), 1e-31)
    assert torch.equal(s, s2) and r_small.psi == pytest.approx(r_small2.psi, rel=1e-12 if dt == np.float64 else 1e-6)
    assert r_small.snorm == pytest.approx(r_small2.snorm, rel=1e-12)
    # offsets rewritten after construction: still n == ngroups m, but two neighbours trade elements
    sizes = np.full(ng, m)
    sizes[10] -= 3; sizes[11] += 3
    offs2 = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    psi._offs.copy_(T(offs2))
    _check(psi, xk, sj, grad, offs2, lam_g, dt)
    # n == 0
    e = torch.empty(0, dtype=T(grad).dtype, device=DEV)
    h0 = sp.GroupNormL2(T(np.array([1.0], dt)), None, offsets=T(np.array([0, 0])))
    psi0 = sp.shifted(h0, e, DELTA, sp.NormLinf(1.0))
    _, r0 = sp.step_(e.clone(), psi0, e.clone(), NU)
    assert tuple(r0) == (0.0, 0.0, 0.0)
    # one group
    xk, sj, grad, offs, lam_g = _uniform(dt, 256, 1)
    _check(_psi(lam_g, offs, xk, sj), xk, sj, grad, offs, lam_g, dt)


def test_step_binf_s_must_not_alias_grad():
    xk, sj, grad, offs, lam_g = _uniform(np.float64, 64, 100)
    psi = _psi(lam_g, offs, xk, sj)
    tg = T(grad)
    with pytest.raises(ValueError):
        sp.step_(tg, psi, tg, NU)
    # nor overlap it partially: the composed form would overwrite part of ∇f before spx_step_post reads it, the one
    # pass another group's ∇f before or after its CTA reads it
    n = grad.size
    buf = T(np.concatenate([grad, grad]))
    for a, b in ((1, 0), (0, 1)):
        with pytest.raises(ValueError):
            sp.step_(buf[a:a + n], psi, buf[b:b + n], NU)
