"""GPU parity of the fused solver step (SURVEY.md §8f rank 1; include/shiftedprox.h: spx_step_sep_*, spx_step_box_*).

The step is the composition  q = -ν∇f;  s = prox!(ψ, q, ν);  xsy = xk + sj + s;  ψ(s);  ‖s‖₂;  ∇f's  in one pass.
Bars: `s` bit-identical to the stand-alone prox! of the same library AND (for the +,-,*,/ operators) to the oracle;
`xsy` bit-identical to (xk + sj) + s; the three scalars against the oracle's composition -- ψ(s) to 1e-12 / 1e-5
relative (Float64 / Float32: λ·Σ is rounded to R), the Float64 sums to 1e-12 relative to Σ|terms|.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from gpu_util import DEV, N, T, bounds, inputs, orc, sp
from shiftedprox import _lib as L

pytestmark = pytest.mark.gpu

DT = [np.float64, np.float32]
H = {"l1": sp.NormL1, "l0": sp.NormL0, "lhalf": sp.RootNormLhalf}


def scalars_close(res, ref_psi, ref_snorm, ref_gdots, grad, s, dt):
    rel = 1e-12 if dt == np.float64 else 1e-5
    assert res.psi == pytest.approx(ref_psi, rel=rel, abs=1e-300)
    assert res.snorm == pytest.approx(ref_snorm, rel=1e-12)
    mag = float(np.sum(np.abs(grad.astype(np.float64) * s.astype(np.float64)))) + 1e-300
    assert abs(res.gdots - ref_gdots) <= 1e-12 * mag


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("n", [1, 7, 1000, 262_147])
@pytest.mark.parametrize("op", ["l1", "l0", "lhalf"])
@pytest.mark.parametrize("twice", [False, True])
def test_step_separable(dt, n, op, twice):
    xk, sj, grad = inputs(n, dt)
    lam, nu = 0.8, 0.35
    if not twice:
        sj = np.zeros(n, dt)
    psi = sp.shifted(H[op](lam), T(xk))
    if twice:
        psi = sp.shifted(psi, T(sj))
    s = torch.empty(n, dtype=T(grad).dtype, device=DEV)
    xsy = torch.empty_like(s)
    out, res = sp.step_(s, psi, T(grad), nu, xsy=xsy)
    assert out is s
    rs, rxsy, rpsi, rsn, rgd = orc.solver_step(op, xk, sj, grad, lam, nu)
    # the stand-alone prox! of the same library, same q
    q = (dt(-dt(nu)) * grad).astype(dt)
    y = torch.empty_like(s)
    sp.prox_(y, psi, T(q), nu)
    assert np.array_equal(N(s), N(y), equal_nan=True)
    if op != "lhalf":
        assert np.array_equal(N(s), rs, equal_nan=True)
    assert np.array_equal(N(xsy), ((xk + sj) + N(s)).astype(dt))
    # scalars: against the oracle composition evaluated at the GPU's own s (identical to rs unless lhalf)
    gs = N(s)
    ref_psi = orc.value_plain(op, xk, sj, gs, lam)
    g64, s64 = grad.astype(np.float64), gs.astype(np.float64)
    scalars_close(res, ref_psi, float(np.sqrt(np.sum(s64 * s64))), float(np.sum(g64 * s64)), grad, gs, dt)
    assert res.psi == pytest.approx(psi(s), rel=1e-12 if dt == np.float64 else 1e-6, abs=1e-300)
    if op != "lhalf":
        assert rpsi == pytest.approx(ref_psi) and rsn == pytest.approx(res.snorm) and rgd == pytest.approx(res.gdots)
    # xsy is optional
    s2 = torch.empty_like(s)
    _, res2 = sp.step_(s2, psi, T(grad), nu)
    assert torch.equal(s2, s) and tuple(res2) == tuple(res)


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("op", ["l1", "l0", "lhalf"])
@pytest.mark.parametrize("vector_bounds", [True, False])
@pytest.mark.parametrize("selected", [None, "odd"])
def test_step_box(dt, op, vector_bounds, selected):
    n = 65_539
    xk, sj, grad = inputs(n, dt)
    lam, nu = 1.0, 0.1
    if vector_bounds:
        l, u = bounds(n, dt)
        tl, tu = T(l), T(u)
    else:
        l, u = -0.7, 0.9
        tl, tu = l, u
    sel = None if selected is None else range(0, n, 2)
    osel = None if selected is None else np.arange(0, n, 2)
    psi = sp.shifted(sp.shifted(H[op](lam), T(xk), tl, tu, selected=sel), T(sj))
    s = torch.empty(n, dtype=T(grad).dtype, device=DEV)
    xsy = torch.empty_like(s)
    _, res = sp.step_(s, psi, T(grad), nu, xsy=xsy)
    q = (dt(-dt(nu)) * grad).astype(dt)
    y = torch.empty_like(s)
    sp.prox_(y, psi, T(q), nu)
    assert np.array_equal(N(s), N(y), equal_nan=True)
    rs, _, _, _, _ = orc.solver_step(op, xk, sj, grad, lam, nu, l, u, osel)
    if op != "lhalf":
        assert np.array_equal(N(s), rs, equal_nan=True)
    gs = N(s)
    assert np.array_equal(N(xsy), ((xk + sj) + gs).astype(dt))
    ref_psi = orc.value_box(op, xk, sj, gs, l, u, lam, osel)
    assert np.isfinite(ref_psi)  # prox! lands inside the box
    g64, s64 = grad.astype(np.float64), gs.astype(np.float64)
    scalars_close(res, ref_psi, float(np.sqrt(np.sum(s64 * s64))), float(np.sum(g64 * s64)), grad, gs, dt)


def test_step_box_reports_infeasible_shift_as_inf():
    # sj outside the box by more than √eps: prox! clamps s into [l - sj, u - sj], so sj + s stays feasible;
    # an inverted box (l > u, which ShiftedRootNormLhalfBox's constructor does not reject) cannot be satisfied
    n = 1000
    xk, sj, grad = inputs(n)
    psi = sp.shifted(sp.shifted(sp.RootNormLhalf(1.0), T(xk), 0.5, -0.5), T(sj))
    s = torch.empty(n, dtype=torch.float64, device=DEV)
    _, res = sp.step_(s, psi, T(grad), 0.1)
    assert res.psi == np.inf and res.psi == psi(s)


@pytest.mark.parametrize("dt", DT)
def test_step_unaligned_and_empty(dt):
    n = 10_001
    xk, sj, grad = inputs(n + 1, dt)
    psi = sp.shifted(sp.shifted(sp.NormL1(1.0), T(xk)[1:]), T(sj)[1:])
    s = torch.empty(n + 1, dtype=T(grad).dtype, device=DEV)[1:]
    xsy = torch.empty(n + 1, dtype=s.dtype, device=DEV)[1:]
    _, res = sp.step_(s, psi, T(grad)[1:], 0.2, xsy=xsy)
    rs, rxsy, rpsi, rsn, rgd = orc.solver_step("l1", xk[1:], sj[1:], grad[1:], 1.0, 0.2)
    assert np.array_equal(N(s), rs) and np.array_equal(N(xsy), rxsy)
    assert res.psi == pytest.approx(rpsi, rel=1e-5) and res.snorm == pytest.approx(rsn) and res.gdots == pytest.approx(rgd)
    e = torch.empty(0, dtype=s.dtype, device=DEV)
    psi0 = sp.shifted(sp.NormL0(1.0), e)
    _, r0 = sp.step_(e.clone(), psi0, e.clone(), 0.2)
    assert tuple(r0) == (0.0, 0.0, 0.0)


@pytest.mark.parametrize("dt", DT)
def test_step_in_place(dt):
    # s may overwrite the gradient and xsy may overwrite xk (x <- x + s): every element's operands are read
    # before its results are written, as for prox!(y, ψ, y, σ) (test/test_allocs.jl:108)
    n = 100_001
    xk, sj, grad = inputs(n, dt)
    z = np.zeros(n, dt)
    rs, rxsy, rpsi, rsn, rgd = orc.solver_step("l0", xk, z, grad, 0.9, 0.25)
    txk, tg = T(xk), T(grad)
    psi = sp.shifted(sp.NormL0(0.9), txk)
    _, res = sp.step_(tg, psi, tg, 0.25, xsy=txk)
    assert np.array_equal(N(tg), rs) and np.array_equal(N(txk), rxsy)
    assert res.psi == pytest.approx(rpsi, rel=1e-5) and res.snorm == pytest.approx(rsn) and res.gdots == pytest.approx(rgd)
    # an output overlapping an input partially would land on other elements' operands, which another CTA reads
    # before or after the store: refused, through the Python API and the raw ABI alike
    buf = T(np.concatenate([grad, grad]))
    with pytest.raises(ValueError):
        sp.step_(buf[1:n + 1], psi, buf[:n], 0.25)
    with pytest.raises(ValueError):
        sp.step_(torch.empty_like(tg), psi, buf[:n], 0.25, xsy=buf[1:n + 1])
    f = getattr(L.lib(), f"spx_step_sep_{'f64' if dt == np.float64 else 'f32'}")
    f.restype = C.c_int32
    st = f(sp.context(DEV), C.c_int32(L.H_L0), C.c_int64(n), C.c_void_p(buf[1:].data_ptr()), None,
           C.c_void_p(buf[n:].data_ptr()), None, C.c_void_p(buf.data_ptr()), C.c_double(0.9), C.c_double(0.25),
           (C.c_double * 3)())
    assert st == L.SPX_E_INVALID


# ---- the step around a prox! that is not one streaming pass (spx_step_pre_*, the type's prox! in place, spx_step_post_*)
def _composed_cases(dt, n):
    from test_gpu_parity import ragged_offsets

    xk, sj, grad = inputs(n, dt)
    offs = ragged_offsets(120, 1500)
    offs = offs[offs <= n]
    if offs[-1] != n:
        offs = np.concatenate([offs, [n]])
    lam_g = (dt(0.5) + orc.uniform(len(offs) - 1, 12, dt)).astype(dt)
    hg = sp.GroupNormL2(T(lam_g), None, offsets=T(offs))
    y0 = orc.prox_l1b2(xk, sj, (dt(-0.3) * grad).astype(dt), 1.0, 0.3, 1e30)
    full = float(np.linalg.norm((y0 + sj).astype(np.float64)))
    return xk, sj, grad, offs, lam_g, {
        "groupl2": (sp.shifted(sp.shifted(hg, T(xk)), T(sj)),
                    lambda s: orc.value_groupl2(xk, sj, s, offs, lam_g)),
        "groupl2binf": (sp.shifted(sp.shifted(hg, T(xk), 0.5, sp.NormLinf(1.0)), T(sj)),
                        lambda s: orc.value_binf("groupl2", xk, sj, s, 0.5, offs=offs, lam_g=lam_g)),
        "l1b2": (sp.shifted(sp.shifted(sp.NormL1(1.0), T(xk), 0.5 * full, sp.NormL2(1.0)), T(sj)),
                 lambda s: orc.value_l1b2(xk, sj, s, 1.0, 0.5 * full)),
        "indballl0": (sp.shifted(sp.shifted(sp.IndBallL0(777), T(xk)), T(sj)),
                      lambda s: orc.value_plain("indballl0", xk, sj, s, r=777)),
        "indballl0binf": (sp.shifted(sp.shifted(sp.IndBallL0(777), T(xk), 1.0, sp.NormLinf(1.0)), T(sj)),
                          lambda s: orc.value_binf("indballl0", xk, sj, s, 1.0, r=777)),
    }


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("kind", ["groupl2", "groupl2binf", "l1b2", "indballl0", "indballl0binf"])
def test_step_composed_types(dt, kind):
    """step_ of the group, top-r and L1B2 types: s bit-identical to the stand-alone prox! of q = -ν∇f, xsy bit-identical
    to (xk + sj) + s, ψ(s) equal to the type's own ψ(s) and to the oracle's value at that s, ‖s‖ and ∇f's against
    Float64 sums of the result."""
    n, nu = 60_013, 0.3
    xk, sj, grad, offs, lam_g, cases = _composed_cases(dt, n)
    psi, oracle_value = cases[kind]
    s = torch.empty(n, dtype=T(grad).dtype, device=DEV)
    xsy = torch.empty_like(s)
    out, res = sp.step_(s, psi, T(grad), nu, xsy=xsy)
    assert out is s
    q = (dt(-dt(nu)) * grad).astype(dt)
    y = torch.empty_like(s)
    sp.prox_(y, psi, T(q), nu)
    assert np.array_equal(N(s), N(y), equal_nan=True)
    assert np.array_equal(N(xsy), ((xk + sj) + N(s)).astype(dt))
    gs = N(s)
    g64, s64 = grad.astype(np.float64), gs.astype(np.float64)
    ref_psi = oracle_value(gs)
    scalars_close(res, ref_psi, float(np.sqrt(np.sum(s64 * s64))), float(np.sum(g64 * s64)), grad, gs, dt)
    assert res.psi == pytest.approx(psi(s), rel=1e-12 if dt == np.float64 else 1e-6, abs=1e-300)
    # xsy is optional; s must not overlap the gradient, and no output may overlap an input partially
    s2 = torch.empty_like(s)
    _, res2 = sp.step_(s2, psi, T(grad), nu)
    assert torch.equal(s2, s) and tuple(res2) == tuple(res)
    tg = T(grad)
    with pytest.raises(ValueError):
        sp.step_(tg, psi, tg, nu)
    buf = T(np.concatenate([grad, grad]))
    with pytest.raises(ValueError):
        sp.step_(buf[1:n + 1], psi, buf[:n], nu)
    with pytest.raises(ValueError):
        sp.step_(s2, psi, buf[:n], nu, xsy=buf[1:n + 1])
    if kind != "l1b2":  # the composed form writes q into s before prox! reads xk
        with pytest.raises(ValueError):
            sp.step_(psi.xk, psi, tg, nu)
    # x <- x + s: xsy may be ψ's own xk
    sp.step_(s2, psi, tg, nu, xsy=psi.xk)
    assert np.array_equal(N(psi.xk), ((xk + sj) + N(s2)).astype(dt))


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("layout", ["g64", "short_ragged"])
def test_step_groupl2_single_pass_on_short_group_layouts(dt, layout):
    """ShiftedGroupNormL2 with every group <= 256 elements (the C4 shape): spx_step_groupl2_* runs the whole step in the
    one pass of the packed warp rounds.  Same bars as above, the composed form of the same call
    (ShiftedProximableFunction.step_) gives the same s bit for bit, and a layout rewritten after validation so that it
    holds a long group (stale census) is still computed correctly (the kernel flags it and the call is redone the long
    way)."""
    rng = np.random.default_rng(7)
    sizes = np.full(1500, 64) if layout == "g64" else rng.integers(1, 257, 1500)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    n, nu = int(offs[-1]), 0.3
    xk, sj, grad = inputs(n, dt)
    lam_g = (dt(0.5) + orc.uniform(len(sizes), 12, dt)).astype(dt)
    psi = sp.shifted(sp.shifted(sp.GroupNormL2(T(lam_g), None, offsets=T(offs)), T(xk)), T(sj))
    s = torch.empty(n, dtype=T(grad).dtype, device=DEV)
    xsy = torch.empty_like(s)

    def check(offsets, step=type(psi).step_):
        launches0 = sp.launch_count(DEV) if hasattr(sp, "launch_count") else None
        _, res = step(psi, s, T(grad), nu, xsy=xsy)
        q = (dt(-dt(nu)) * grad).astype(dt)
        y = torch.empty_like(s)
        sp.prox_(y, psi, T(q), nu)
        assert np.array_equal(N(s), N(y))
        assert np.array_equal(N(xsy), ((xk + sj) + N(s)).astype(dt))
        gs = N(s)
        g64, s64 = grad.astype(np.float64), gs.astype(np.float64)
        scalars_close(res, orc.value_groupl2(xk, sj, gs, offsets, lam_g), float(np.sqrt(np.sum(s64 * s64))),
                      float(np.sum(g64 * s64)), grad, gs, dt)
        return res, launches0

    res, _ = check(offs)
    s_fused = s.clone()
    res_c, _ = check(offs, sp.ShiftedProximableFunction.step_)
    assert torch.equal(s, s_fused)
    assert res_c.psi == pytest.approx(res.psi, rel=1e-12 if dt == np.float64 else 1e-6)
    assert res_c.snorm == pytest.approx(res.snorm, rel=1e-12) and res_c.gdots == pytest.approx(res.gdots, rel=1e-9, abs=1e-9)
    # stale census: same address, ngroups and n, but two neighbours merged into one long group and one group split
    new = sizes.copy()
    big = int(np.argmax(np.cumsum(new) > n // 2))
    take = 0
    j = big + 1
    while new[big] + take <= 300:
        take += new[j]; new[j] = 0; j += 1
    new[big] += take
    offs2 = np.concatenate([[0], np.cumsum(new)]).astype(np.int64)
    assert offs2[-1] == n and np.max(new) > 256
    psi._offs.copy_(T(offs2))
    check(offs2)
