"""GPU parity of the fused step around iprox! (include/shiftedprox.h: spx_istep_sep_*, spx_istep_box_*).

The step is the composition  d = D + σ;  s = iprox!(ψ, ∇f, d);  xsy = xk + sj + s;  ψ(s);  ‖s‖₂;  ∇f's;  sᵀ d s  in one
pass of step_kernel.  Bars: `s` bit-identical to the stand-alone iprox! of the same library at d = D + σ rounded to R,
and to the oracle; `xsy` bit-identical to (xk + sj) + s; ψ(s), ‖s‖ and ∇f·s as in test_gpu_step.py; sᵀ d s to 1e-12 of
Σ|d s²| against Float64 numpy at the GPU's own s.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from gpu_util import DEV, N, T, bounds, diag, inputs, orc, sp
from istep_oracle import solver_istep
from test_gpu_step import scalars_close

pytestmark = pytest.mark.gpu

DT = [np.float64, np.float32]
H = {"l1": sp.NormL1, "l0": sp.NormL0}


def positive_diag(n, dt):
    return orc.uniform(n, 5, dt, 1.0, 0.5)  # 0.5 + u


def shifted_d(D, dshift):
    """D .+ σ as the caller's broadcast rounds it"""
    return (D + D.dtype.type(dshift)).astype(D.dtype)


def sds_close(res, s, d):
    s64, d64 = s.astype(np.float64), d.astype(np.float64)
    terms = d64 * s64 * s64
    assert abs(res.sds - float(np.sum(terms))) <= 1e-12 * (float(np.sum(np.abs(terms))) + 1e-300)


def same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("n", [1, 7, 1000, 262_147])
@pytest.mark.parametrize("op", ["l1", "l0"])
@pytest.mark.parametrize("twice", [False, True])
@pytest.mark.parametrize("dshift", [0.0, 0.25])
def test_istep_separable(dt, n, op, twice, dshift):
    xk, sj, grad = inputs(n, dt)
    D = positive_diag(n, dt)
    lam = 0.8
    if not twice:
        sj = np.zeros(n, dt)
    psi = sp.shifted(H[op](lam), T(xk))
    if twice:
        psi = sp.shifted(psi, T(sj))
    s = torch.empty(n, dtype=T(grad).dtype, device=DEV)
    xsy = torch.empty_like(s)
    out, res = sp.istep_(s, psi, T(grad), T(D), dshift, xsy=xsy)
    assert out is s and isinstance(res, sp.IStepResult)
    d = shifted_d(D, dshift)
    y = torch.empty_like(s)
    sp.iprox_(y, psi, T(grad), T(d))
    gs = N(s)
    assert same_bits(gs, N(y))
    rs, rxsy, rpsi, rsn, rgd, rsds = solver_istep(op, xk, sj, grad, D, dshift, lam)
    assert same_bits(gs, rs)
    assert same_bits(N(xsy), ((xk + sj) + gs).astype(dt))
    g64, s64 = grad.astype(np.float64), gs.astype(np.float64)
    scalars_close(res, orc.value_plain(op, xk, sj, gs, lam), float(np.sqrt(np.sum(s64 * s64))),
                  float(np.sum(g64 * s64)), grad, gs, dt)
    sds_close(res, gs, d)
    assert rpsi == pytest.approx(res.psi) and rsn == pytest.approx(res.snorm) and rgd == pytest.approx(res.gdots)
    assert rsds == pytest.approx(res.sds)
    # xsy is optional
    s2 = torch.empty_like(s)
    _, res2 = sp.istep_(s2, psi, T(grad), T(D), dshift)
    assert torch.equal(s2, s) and tuple(res2) == tuple(res)


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("op", ["l1", "l0"])
@pytest.mark.parametrize("vector_bounds", [True, False])
@pytest.mark.parametrize("selected", [None, "even"])
@pytest.mark.parametrize("dshift", [0.0, 0.25])
def test_istep_box(dt, op, vector_bounds, selected, dshift):
    n = 65_539
    xk, sj, grad = inputs(n, dt)
    D = diag(n, dt)  # 80 % positive, 10 % negative, 10 % exactly 0
    lam = 1.0
    if vector_bounds:
        l, u = bounds(n, dt)
        tl, tu = T(l), T(u)
    else:
        l, u = -0.7, 0.9
        tl, tu = l, u
    sel = range(0, n, 2) if selected else None
    sel_host = np.arange(0, n, 2) if selected else None
    psi = sp.shifted(sp.shifted(H[op](lam), T(xk), tl, tu, sel), T(sj))
    s = torch.empty(n, dtype=T(grad).dtype, device=DEV)
    xsy = torch.empty_like(s)
    _, res = sp.istep_(s, psi, T(grad), T(D), dshift, xsy=xsy)
    d = shifted_d(D, dshift)
    y = torch.empty_like(s)
    sp.iprox_(y, psi, T(grad), T(d))
    gs = N(s)
    assert same_bits(gs, N(y))
    rs, _, rpsi, _, _, rsds = solver_istep(op, xk, sj, grad, D, dshift, lam, l, u, sel_host)
    assert same_bits(gs, rs)
    assert same_bits(N(xsy), ((xk + sj) + gs).astype(dt))
    ref_psi = orc.value_box(op, xk, sj, gs, l, u, lam, sel_host)
    g64, s64 = grad.astype(np.float64), gs.astype(np.float64)
    scalars_close(res, ref_psi, float(np.sqrt(np.sum(s64 * s64))), float(np.sum(g64 * s64)), grad, gs, dt)
    assert res.psi == pytest.approx(psi(s), rel=1e-12 if dt == np.float64 else 2e-6, abs=1e-300)
    sds_close(res, gs, d)
    assert rpsi == pytest.approx(res.psi) and rsds == pytest.approx(res.sds)


@pytest.mark.parametrize("op", ["l1", "l0"])
def test_istep_box_infeasible_shift(op):
    """ψ(s) is Inf when sj + s cannot lie in [l - ϵ, u + ϵ]: iprox! keeps s in [l - sj, u - sj], so only an inverted
    box (set_bounds! does not check l <= u) makes the step infeasible"""
    n = 4099
    xk, sj, grad = inputs(n, np.float64)
    D = positive_diag(n, np.float64)
    psi = sp.shifted(sp.shifted(H[op](1.0), T(xk), -1.0, 1.0, range(0, n, 2)), T(sj))
    sp.set_bounds_(psi, 0.5, -0.5)
    s = torch.empty(n, dtype=torch.float64, device=DEV)
    _, res = sp.istep_(s, psi, T(grad), T(D), 0.1)
    assert res.psi == np.inf and psi(s) == np.inf
    assert orc.value_box(op, xk, sj, N(s), 0.5, -0.5, 1.0, np.arange(0, n, 2)) == np.inf


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("op", ["l1", "l0"])
def test_istep_box_special_values(dt, op):
    """NaN / ±Inf / ±0 operands and d next to ±eps: s is still the stand-alone iprox!'s, and the oracle's except on the
    documented L0Box NaN corner (test_gpu_bulk_stream.py::test_bulk_box_iprox)"""
    from test_gpu_bulk_stream import _operands
    n = 70_001
    xk, sj, g, l, u, D = _operands(n, dt, special=True)
    lam = 0.8
    psi = sp.shifted(sp.shifted(H[op](lam), T(xk), T(l), T(u)), T(sj))
    s = torch.empty(n, dtype=T(g).dtype, device=DEV)
    xsy = torch.empty_like(s)
    _, res = sp.istep_(s, psi, T(g), T(D), 0.0, xsy=xsy)
    d = shifted_d(D, 0.0)
    y = torch.empty_like(s)
    _, v = sp.iprox_(y, psi, T(g), T(d), want_value=True)
    gs = N(s)
    assert same_bits(gs, N(y))
    # NaN payloads of the device sums need not be numpy's
    with np.errstate(invalid="ignore"):
        assert np.array_equal(N(xsy), ((xk + sj) + gs).astype(dt), equal_nan=True)
    ref = orc.iprox_box(op, xk, sj, g, d, l, u, lam)
    keep = np.ones(n, bool)
    if op == "l0":
        keep = ~(np.isnan(xk) | np.isnan(sj) | np.isnan(g) | np.isnan(d) | np.isnan(l) | np.isnan(u))
    assert np.array_equal(gs[keep], ref[keep], equal_nan=True)
    assert (np.isnan(res.psi) and np.isnan(v)) or res.psi == pytest.approx(v, rel=1e-12 if dt == np.float64 else 2e-6)


@pytest.mark.parametrize("dt", DT)
def test_istep_across_kernels(dt):
    """Vector-bound L0Box at n >= 2^20: the stand-alone iprox! runs in ew_bulk_kernel, the istep in step_kernel"""
    from torch.profiler import ProfilerActivity, profile
    n = (1 << 20) + 333
    xk, sj, grad = inputs(n, dt)
    l, u = bounds(n, dt)
    D = diag(n, dt)
    psi = sp.shifted(sp.shifted(sp.NormL0(0.8), T(xk), T(l), T(u)), T(sj))
    s = torch.empty(n, dtype=T(grad).dtype, device=DEV)
    y = torch.empty_like(s)
    tg, tD = T(grad), T(D)
    d = shifted_d(D, 0.25)
    td = T(d)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(2):  # twice: the first activity of a profiling window can go unrecorded
            sp.istep_(s, psi, tg, tD, 0.25)
            sp.iprox_(y, psi, tg, td)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert any("step_kernel" in k for k in names) and any("ew_bulk_kernel" in k for k in names), names
    assert same_bits(N(s), N(y))
    assert same_bits(N(s), orc.iprox_box("l0", xk, sj, grad, d, l, u, 0.8))


@pytest.mark.parametrize("op", ["l1", "l0"])
@pytest.mark.parametrize("twice", [False, True])
def test_istep_assertion(op, twice):
    n, k = 10_007, 4_321
    xk, sj, grad = inputs(n, np.float64)
    D = positive_diag(n, np.float64)
    D[k] = -0.3
    psi = sp.shifted(H[op](1.0), T(xk))
    if twice:
        psi = sp.shifted(psi, T(sj))
    s = torch.zeros(n, dtype=torch.float64, device=DEV)
    with pytest.raises(AssertionError, match=rf"d\[{k}\]"):
        sp.istep_(s, psi, T(grad), T(D))
    # s is still written in full, as by the stand-alone iprox!
    y = torch.zeros_like(s)
    with pytest.raises(AssertionError, match=rf"d\[{k}\]"):
        sp.iprox_(y, psi, T(grad), T(D))
    assert same_bits(N(s), N(y))
    # a shift that makes every d positive passes
    _, res = sp.istep_(s, psi, T(grad), T(D), 0.5)
    y2 = torch.empty_like(s)
    sp.iprox_(y2, psi, T(grad), T(shifted_d(D, 0.5)))
    assert same_bits(N(s), N(y2)) and np.isfinite(res.sds)


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("box", [False, True])
def test_istep_unaligned_views(dt, box):
    n = 100_003
    xk, sj, grad = inputs(n + 1, dt)
    D = positive_diag(n + 1, dt)
    l, u = bounds(n + 1, dt)

    def run(sl):
        h = sp.NormL1(0.7)
        psi = sp.shifted(h, T(xk)[sl], T(l)[sl], T(u)[sl]) if box else sp.shifted(h, T(xk)[sl])
        psi = sp.shifted(psi, T(sj)[sl])
        s = torch.empty(n + 1, dtype=T(grad).dtype, device=DEV)[sl]
        xsy = torch.empty(n + 1, dtype=T(grad).dtype, device=DEV)[sl]
        _, res = sp.istep_(s, psi, T(grad)[sl], T(D)[sl], 0.25, xsy=xsy)
        return N(s), N(xsy), res

    s_off, xsy_off, r_off = run(slice(1, None))  # operands one element past the 16-byte grid: the scalar loop
    s_al, xsy_al, _ = run(slice(0, n))       # the first n elements, aligned: the vector loop
    rs, rxsy, _, _, _, _ = solver_istep("l1", xk[1:], sj[1:], grad[1:], D[1:], 0.25, 0.7,
                                        *((l[1:], u[1:]) if box else ()))
    assert same_bits(s_off, rs) and same_bits(xsy_off, rxsy)
    rs, rxsy, _, _, _, _ = solver_istep("l1", xk[:n], sj[:n], grad[:n], D[:n], 0.25, 0.7,
                                        *((l[:n], u[:n]) if box else ()))
    assert same_bits(s_al, rs) and same_bits(xsy_al, rxsy)
    # the sums of the two loops fold in different orders
    _, _, rpsi, rsn, rgd, rsds = solver_istep("l1", xk[1:], sj[1:], grad[1:], D[1:], 0.25, 0.7,
                                              *((l[1:], u[1:]) if box else ()))
    for a, b in zip(r_off, (rpsi, rsn, rgd, rsds)):
        assert a == pytest.approx(b, rel=1e-12 if dt == np.float64 else 1e-5)


@pytest.mark.parametrize("box", [False, True])
def test_istep_empty(box):
    e = torch.empty(0, dtype=torch.float64, device=DEV)
    psi = sp.shifted(sp.NormL0(1.0), e, e, e) if box else sp.shifted(sp.NormL0(1.0), e)
    _, res = sp.istep_(torch.empty(0, dtype=torch.float64, device=DEV), psi, e, e, 0.5, xsy=e)
    assert tuple(res) == (0.0, 0.0, 0.0, 0.0)


@pytest.mark.parametrize("op", ["l1", "l0"])
@pytest.mark.parametrize("box", [False, True])
def test_istep_in_place_and_deterministic(op, box):
    """s = grad and xsy = xk: each element's operands are read before its results are written"""
    n = 262_147
    xk, sj, grad = inputs(n, np.float64)
    D = diag(n, np.float64) if box else positive_diag(n, np.float64)
    l, u = bounds(n, np.float64)

    def make(txk):
        psi = sp.shifted(H[op](0.9), txk, T(l), T(u)) if box else sp.shifted(H[op](0.9), txk)
        return sp.shifted(psi, T(sj))

    s, xsy = torch.empty(n, dtype=torch.float64, device=DEV), torch.empty(n, dtype=torch.float64, device=DEV)
    _, ref = sp.istep_(s, make(T(xk)), T(grad), T(D), 0.25, xsy=xsy)
    for _ in range(3):
        _, again = sp.istep_(torch.empty_like(s), make(T(xk)), T(grad), T(D), 0.25)
        assert np.asarray(tuple(again)).tobytes() == np.asarray(tuple(ref)).tobytes()
    txk, tg = T(xk), T(grad)
    _, r = sp.istep_(tg, make(txk), tg, T(D), 0.25, xsy=txk)
    assert torch.equal(tg, s) and torch.equal(txk, xsy)
    assert np.asarray(tuple(r)).tobytes() == np.asarray(tuple(ref)).tobytes()


def test_istep_rejections():
    n = 1000
    xk, sj, grad = inputs(n, np.float64)
    l, u = bounds(n, np.float64)
    txk, tg, tD = T(xk), T(grad), T(positive_diag(n, np.float64))
    s = torch.empty_like(tg)
    for psi in (sp.shifted(sp.RootNormLhalf(1.0), txk), sp.shifted(sp.RootNormLhalf(1.0), txk, T(l), T(u))):
        with pytest.raises(NotImplementedError):
            sp.istep_(s, psi, tg, tD)
    # through the C ABI: no iprox! for RootNormLhalf and its Box form
    lib = sp.L.lib()
    out = (C.c_double * 4)()
    bad = C.c_int64()
    ctx = sp.context(DEV)
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    lib.spx_istep_sep_f64.restype = C.c_int32
    st = lib.spx_istep_sep_f64(ctx, C.c_int32(sp.L.H_LHALF), C.c_int64(n), p(s), None, p(txk), None, p(tg), p(tD),
                               C.c_double(0.0), C.c_double(1.0), C.byref(bad), out)
    assert st == sp.L.SPX_E_INVALID
    tl = T(l)
    lb, ub = sp.L.Bound(tl.data_ptr(), 0.0), sp.L.Bound(None, 1.0)
    sel = sp.L.Sel(sp.L.SEL_ALL, 0, 1, n - 1, None, None, 0)
    lib.spx_istep_box_f64.restype = C.c_int32
    st = lib.spx_istep_box_f64(ctx, C.c_int32(sp.L.BOX_LHALF), C.c_int64(n), p(s), None, p(txk), p(txk), p(tg), p(tD),
                               C.c_double(0.0), C.byref(lb), C.byref(ub), C.byref(sel), C.c_double(1.0), out)
    assert st == sp.L.SPX_E_INVALID
