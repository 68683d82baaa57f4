"""GPU tests of the ShiftedNormL1B2 solver step (include/shiftedprox.h: spx_step_l1b2_*, spx_step_l1b2_sharded_*).

The step runs inside the passes of prox!'s own root search: every pass forms q = fl(-ν∇f) from ∇f, the finish writes
s and xsy = (xk + sj) + s and sums ψ(s), Σs², Σ∇f·s.  Bars:
  * s bit-identical to the stand-alone prox_(y, ψ, fl(-ν∇f), ν) into a y that overlaps no input, with the same pass
    count and the same number of launches (no pre or post pass); within the L1B2 bar of the oracle (64 / 16 ulp of
    |ref| + |sj| + 1) and ‖sj + s‖ = Δ (1e-10 / 1e-5) when the ball is active;
  * xsy bit-identical to (xk + sj) + s;
  * ψ(s) against the oracle's value at the GPU's s and against ψ(s) of the library (1e-12 / 1e-5 relative), Σs² to
    1e-12 relative and Σ∇f·s to 1e-12 of Σ|∇f s| against Float64 sums;
  * with xsy aliasing xk (x <- x + s) no pass stashes and the finish checks no unverified root: s and the pass count
    are those of the in-place prox_(s, ψ, s, ν).
The finish runs on step_kernel's grid, which can differ from the prox! finish's (Float32 at large n): Σ(sj + s)², the
check of an unverified root, is then summed in another order.  The parity grid includes those sizes.
SPX_FULLSIZE=0 runs the C3-sized case as Float64 2^27 instead of Float32 2^29.
"""
import ctypes as C
import math
import os
import threading

import numpy as np
import pytest
import torch

from gpu_util import DEV, N, T, inputs, orc, sp
from shiftedprox import _lib as L

pytestmark = pytest.mark.gpu

DT = [np.float64, np.float32]
FULL = os.environ.get("SPX_FULLSIZE", "1") != "0"
LAM, NU = 1.0, 0.3


def eps(dt):
    return float(np.finfo(dt).eps)


def bits_equal(a, b):
    a, b = np.asarray(a), np.asarray(b)
    it = np.uint64 if a.dtype == np.float64 else np.uint32
    return a.shape == b.shape and bool(np.all((a.view(it) == b.view(it)) | (np.isnan(a) & np.isnan(b))))


def mnu_q(grad, dt):
    """fl(-ν ∇f) in R, as the caller's broadcast rounds it"""
    return (dt(-dt(NU)) * grad).astype(dt)


def full_norm(xk, sj, q, dt):
    y0 = orc.prox_l1b2(xk, sj, q, LAM, NU, 1e30)  # ball inactive
    return float(np.linalg.norm((y0 + sj).astype(np.float64)))


def make_psi(xk, sj, delta, twice):
    psi = sp.shifted(sp.NormL1(LAM), T(xk), delta, sp.NormL2(1.0))
    return sp.shifted(psi, T(sj)) if twice else psi


def counted(fn):
    l0 = sp.launch_count(DEV)
    r = fn()
    return r, sp.launch_count(DEV) - l0


def check_scalars(res, psi, s, grad, xk, sj, delta, dt):
    gs = N(s)
    rel = 1e-12 if dt == np.float64 else 1e-5
    assert res.psi == pytest.approx(orc.value_l1b2(xk, sj, gs, LAM, delta), rel=rel, abs=1e-300)
    assert res.psi == pytest.approx(psi(s), rel=rel, abs=1e-300)
    g64, s64 = grad.astype(np.float64), gs.astype(np.float64)
    assert res.snorm ** 2 == pytest.approx(float(np.sum(s64 * s64)), rel=1e-12, abs=1e-300)
    assert abs(res.gdots - float(np.sum(g64 * s64))) <= 1e-12 * (float(np.sum(np.abs(g64 * s64))) + 1e-300)


def check_against_oracle(gs, xk, sj, q, delta, full, dt):
    ref = orc.prox_l1b2(xk, sj, q, LAM, NU, delta)
    tol = (64 if dt == np.float64 else 16) * eps(dt) * (np.abs(ref) + np.abs(sj) + 1)
    assert np.array_equal(np.isnan(gs), np.isnan(ref))
    ok = ~np.isnan(ref)
    assert np.all(np.abs(gs[ok].astype(np.float64) - ref[ok].astype(np.float64)) <= tol[ok])
    if delta < full:
        nrm = float(np.linalg.norm((gs + sj).astype(np.float64)))
        assert nrm == pytest.approx(delta, rel=1e-10 if dt == np.float64 else 1e-5)


# ------------------------------------------------------------------------------------------------ parity ---
@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("n", [5, 1000, 262_147, (1 << 22) + 3])
@pytest.mark.parametrize("frac", [2.0, 0.5, 0.01])
@pytest.mark.parametrize("twice", [False, True])
def test_step_l1b2_matches_prox(dt, n, frac, twice):
    xk, sj, grad = inputs(n, dt)
    if not twice:
        sj = np.zeros(n, dt)
    q = mnu_q(grad, dt)
    full = full_norm(xk, sj, q, dt)
    delta = frac * full
    psi = make_psi(xk, sj, delta, twice)
    tg = T(grad)
    s = torch.empty(n, dtype=tg.dtype, device=DEV)
    xsy = torch.empty_like(s)
    (out, res), nl_step = counted(lambda: sp.step_(s, psi, tg, NU, xsy=xsy))
    assert out is s
    passes = psi.last_passes
    # the stand-alone prox! of fl(-ν∇f) into a disjoint y, its ψ folded like the step's
    y = torch.empty_like(s)
    (_, val), nl_prox = counted(lambda: sp.prox_(y, psi, T(q), NU, want_value=True))
    assert bits_equal(N(s), N(y))
    assert passes == psi.last_passes
    assert nl_step == nl_prox  # no pre or post pass
    gs = N(s)
    assert bits_equal(N(xsy), ((xk + sj) + gs).astype(dt))
    check_against_oracle(gs, xk, sj, q, delta, full, dt)
    check_scalars(res, psi, s, grad, xk, sj, delta, dt)
    assert res.psi == pytest.approx(val, rel=1e-12 if dt == np.float64 else 1e-6, abs=1e-300)
    # without xsy: same s and scalars; three identical calls: identical scalars
    s2 = torch.empty_like(s)
    _, res2 = sp.step_(s2, psi, tg, NU)
    assert torch.equal(s2, s) and tuple(res2) == tuple(res)
    for _ in range(2):
        _, r = sp.step_(s2, psi, tg, NU, xsy=xsy)
        assert tuple(r) == tuple(res)


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("frac", [0.5, 1e9])
def test_step_l1b2_nan_in_xk_gives_what_prox_gives(dt, frac):
    """A NaN in xk makes every norm of the search NaN: the step gives what prox_ gives, NaN positions included."""
    n = 50_001
    xk, sj, grad = inputs(n, dt)
    q = mnu_q(grad, dt)
    full = full_norm(xk, sj, q, dt)
    xk = xk.copy()
    xk[12345] = np.nan
    delta = frac * full if frac < 1e6 else 1e30
    psi = make_psi(xk, sj, delta, True)
    s = torch.empty(n, dtype=T(grad).dtype, device=DEV)
    sp.step_(s, psi, T(grad), NU)
    passes = psi.last_passes
    y = torch.empty_like(s)
    sp.prox_(y, psi, T(q), NU)
    assert bits_equal(N(s), N(y)) and passes == psi.last_passes
    ref = orc.prox_l1b2(xk, sj, q, LAM, NU, delta)
    got = N(s)
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    ok = ~np.isnan(ref)
    assert np.all(np.abs(got[ok].astype(np.float64) - ref[ok].astype(np.float64)) <= 64 * eps(dt) * (np.abs(ref[ok]) + 1))


# ---------------------------------------------------------------------------------------------- aliasing ---
@pytest.mark.parametrize("dt", DT)
def test_step_l1b2_s_overlapping_grad_is_refused(dt):
    n = 1000
    xk, sj, grad = inputs(n, dt)
    psi = make_psi(xk, sj, 1.0, True)
    buf = T(np.concatenate([grad, grad]))
    with pytest.raises(ValueError):
        sp.step_(buf[:n], psi, buf[:n], NU)
    with pytest.raises(ValueError):
        sp.step_(buf[1:n + 1], psi, buf[:n], NU)
    out, passes = (C.c_double * 3)(), C.c_int32()
    suf = "f64" if dt == np.float64 else "f32"
    f = getattr(L.lib(), f"spx_step_l1b2_{suf}")
    f.restype = C.c_int32
    for a, b in ((0, 0), (1, 0), (0, 1)):
        st = f(sp.context(DEV), C.c_int64(n), C.c_void_p(buf[a:].data_ptr()), None, C.c_void_p(psi.xk.data_ptr()),
               C.c_void_p(psi.sj.data_ptr()), C.c_void_p(buf[b:].data_ptr()), C.c_double(LAM), C.c_double(NU),
               C.c_double(1.0), C.c_double(1.0), C.byref(passes), out)
        assert st == L.SPX_E_INVALID


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("n", [262_147, (1 << 22) + 3])
def test_step_l1b2_xsy_aliasing_xk_takes_the_in_place_route(dt, n):
    """x <- x + s: xsy is ψ.xk itself.  No pass stashes and the finish checks no unverified root, so s and the pass
    count are those of the in-place prox_(s, ψ, s, ν) (s pre-filled with q), and xsy = old xk + sj + s."""
    xk, sj, grad = inputs(n, dt)
    q = mnu_q(grad, dt)
    delta = 0.5 * full_norm(xk, sj, q, dt)
    ref_psi = make_psi(xk, sj, delta, True)
    y = T(q).clone()
    sp.prox_(y, ref_psi, y, NU)
    ref_passes = ref_psi.last_passes
    psi = make_psi(xk, sj, delta, True)
    s = torch.empty_like(y)
    _, res = sp.step_(s, psi, T(grad), NU, xsy=psi.xk)
    assert bits_equal(N(s), N(y))
    assert psi.last_passes == ref_passes
    assert bits_equal(N(psi.xk), ((xk + sj) + N(s)).astype(dt))
    check_against_oracle(N(s), xk, sj, q, delta, 2 * delta, dt)
    g64, s64 = grad.astype(np.float64), N(s).astype(np.float64)
    assert res.snorm ** 2 == pytest.approx(float(np.sum(s64 * s64)), rel=1e-12)
    assert abs(res.gdots - float(np.sum(g64 * s64))) <= 1e-12 * float(np.sum(np.abs(g64 * s64)))


@pytest.mark.parametrize("dt", DT)
def test_step_l1b2_xsy_overlapping_s_is_refused(dt):
    """s holds the search's stash of sj + q while the finish writes xsy: an xsy that overlaps s is refused."""
    n = 1000
    xk, sj, grad = inputs(n, dt)
    psi = make_psi(xk, sj, 1.0, True)
    tg = T(grad)
    buf = torch.empty(2 * n, dtype=tg.dtype, device=DEV)
    for a in (0, 1):
        with pytest.raises(ValueError):
            sp.step_(buf[:n], psi, tg, NU, xsy=buf[a:a + n])
    out, passes = (C.c_double * 3)(), C.c_int32()
    f = getattr(L.lib(), f"spx_step_l1b2_{'f64' if dt == np.float64 else 'f32'}")
    f.restype = C.c_int32
    for a in (0, 1):
        st = f(sp.context(DEV), C.c_int64(n), C.c_void_p(buf.data_ptr()), C.c_void_p(buf[a:].data_ptr()),
               C.c_void_p(psi.xk.data_ptr()), C.c_void_p(psi.sj.data_ptr()), C.c_void_p(tg.data_ptr()),
               C.c_double(LAM), C.c_double(NU), C.c_double(1.0), C.c_double(1.0), C.byref(passes), out)
        assert st == L.SPX_E_INVALID


@pytest.mark.parametrize("dt", DT)
def test_step_l1b2_unaligned_views_match_prox(dt):
    """Every vector one element into its buffer (not 16-byte aligned): the VEC = 1 instances of the GRAD norm passes
    and of the step's finish, against the prox! of the same offset views."""
    n = 262_147
    xk, sj, grad = inputs(n + 1, dt)
    q = mnu_q(grad, dt)
    delta = 0.5 * full_norm(xk[1:], sj[1:], q[1:], dt)
    psi = sp.shifted(sp.shifted(sp.NormL1(LAM), T(xk)[1:], delta, sp.NormL2(1.0)), T(sj)[1:])
    assert psi.xk.data_ptr() % 16 != 0
    tg = T(grad)[1:]
    s = torch.empty(n + 1, dtype=tg.dtype, device=DEV)[1:]
    xsy = torch.empty(n + 1, dtype=tg.dtype, device=DEV)[1:]
    _, res = sp.step_(s, psi, tg, NU, xsy=xsy)
    passes = psi.last_passes
    y = torch.empty(n + 1, dtype=tg.dtype, device=DEV)[1:]
    sp.prox_(y, psi, T(q)[1:], NU)
    assert bits_equal(N(s), N(y)) and passes == psi.last_passes
    assert bits_equal(N(xsy), ((xk[1:] + sj[1:]) + N(s)).astype(dt))
    check_against_oracle(N(s), xk[1:], sj[1:], q[1:], delta, 2 * delta, dt)
    check_scalars(res, psi, s, grad[1:], xk[1:], sj[1:], delta, dt)


@pytest.mark.parametrize("dt", DT)
def test_step_l1b2_empty(dt):
    e = torch.empty(0, dtype=torch.float64 if dt == np.float64 else torch.float32, device=DEV)
    psi = sp.shifted(sp.NormL1(LAM), e, 1.0, sp.NormL2(1.0))
    _, r = sp.step_(e.clone(), psi, e.clone(), NU, xsy=e.clone())
    assert tuple(r) == (0.0, 0.0, 0.0)


# ---------------------------------------------------------------------------------------------- sharded ---
def call_sharded(ctx, suf, n, s, xsy, xk, sj, g, delta, cb, passes, out):
    L.call(f"spx_step_l1b2_sharded_{suf}", ctx, C.c_int64(n), C.c_void_p(s.data_ptr()),
           C.c_void_p(xsy.data_ptr() if xsy is not None else 0), C.c_void_p(xk.data_ptr()), C.c_void_p(sj.data_ptr()),
           C.c_void_p(g.data_ptr()), C.c_double(LAM), C.c_double(NU), C.c_double(delta), C.c_double(1.0), cb, None,
           C.byref(passes), out)


@pytest.mark.parametrize("dt", DT)
def test_step_l1b2_sharded_identity_callback_gives_the_unsharded_bits(dt):
    n = 200_001
    xk, sj, grad = inputs(n, dt)
    delta = 0.5 * full_norm(xk, sj, mnu_q(grad, dt), dt)
    psi = make_psi(xk, sj, delta, True)
    tg = T(grad)
    s1, x1 = torch.empty_like(tg), torch.empty_like(tg)
    _, res = sp.step_(s1, psi, tg, NU, xsy=x1)
    calls = []

    def ident(_u, vals, count):  # world size 1: the all-reduce is the identity
        calls.append(count)
        return 0

    s2, x2 = torch.empty_like(tg), torch.empty_like(tg)
    out, passes = (C.c_double * 3)(), C.c_int32()
    call_sharded(sp.context(DEV), "f64" if dt == np.float64 else "f32", n, s2, x2, psi.xk, psi.sj, tg, delta,
                 L.ALLREDUCE_FN(ident), passes, out)
    assert torch.equal(s1, s2) and torch.equal(x1, x2)
    assert passes.value == psi.last_passes and len(calls) == passes.value
    assert calls[-1] == 4 and all(c % 2 == 0 for c in calls)
    assert (out[0], math.sqrt(out[1]), out[2]) == tuple(res)


@pytest.mark.parametrize("dt", DT)
def test_step_l1b2_sharded_wrapper_on_one_rank(dt, tmp_path):
    """sharded.step_l1b2_sharded_ over a torch.distributed group of one rank (gloo, file store): the wrapper's
    all-reduce callback runs on every pass and the result is the unsharded step's, bit for bit."""
    import torch.distributed as dist

    from shiftedprox import sharded

    n = 100_003
    xk, sj, grad = inputs(n, dt)
    delta = 0.5 * full_norm(xk, sj, mnu_q(grad, dt), dt)
    psi = make_psi(xk, sj, delta, True)
    tg = T(grad)
    s1, x1 = torch.empty_like(tg), torch.empty_like(tg)
    _, res = sp.step_(s1, psi, tg, NU, xsy=x1)
    passes = psi.last_passes
    dist.init_process_group("gloo", store=dist.FileStore(str(tmp_path / "store"), 1), rank=0, world_size=1)
    try:
        s2, x2 = torch.empty_like(tg), torch.empty_like(tg)
        out, res2 = sharded.step_l1b2_sharded_(s2, psi, tg, NU, xsy_local=x2)
    finally:
        dist.destroy_process_group()
    assert out is s2
    assert torch.equal(s1, s2) and torch.equal(x1, x2)
    assert psi.last_passes == passes and tuple(res2) == tuple(res)


@pytest.mark.parametrize("dt", DT)
def test_step_l1b2_over_two_shards(dt):
    """One vector cut into two shards (two contexts with their own streams, two host threads standing in for two
    ranks; the all-reduce callback meets at a barrier): both ranks return the same out3 and pass count, and the
    concatenated s is the single-device step's to the L1B2 bar."""
    n = 300_001
    xk, sj, grad = inputs(n, dt)
    delta = 0.5 * full_norm(xk, sj, mnu_q(grad, dt), dt)
    psi = make_psi(xk, sj, delta, True)
    s_one = torch.empty(n, dtype=T(grad).dtype, device=DEV)
    _, res = sp.step_(s_one, psi, T(grad), NU)
    world, cut = 2, (n // 2 + 3) & ~3
    bounds_ = [(0, cut), (cut, n)]
    suf = "f64" if dt == np.float64 else "f32"
    barrier = threading.Barrier(world)
    slots, outs, errs = [None] * world, [None] * world, []

    def worker(rank):
        try:
            lo, hi = bounds_[rank]
            ctx = C.c_void_p()
            L.call("spx_ctx_create", C.byref(ctx), C.c_int32(0), C.c_void_p(0), C.c_int32(1))
            txk, tsj, tg = T(xk[lo:hi]), T(sj[lo:hi]), T(grad[lo:hi])
            s, xsy = torch.empty_like(tg), torch.empty_like(tg)
            torch.cuda.synchronize()

            def reduce(_user, vals, count):
                slots[rank] = [vals[i] for i in range(count)]
                barrier.wait()
                tot = [sum(sl[i] for sl in slots) for i in range(count)]
                barrier.wait()
                for i in range(count):
                    vals[i] = tot[i]
                return 0

            out, passes = (C.c_double * 3)(), C.c_int32()
            call_sharded(ctx, suf, hi - lo, s, xsy, txk, tsj, tg, delta, L.ALLREDUCE_FN(reduce), passes, out)
            L.call("spx_ctx_synchronize", ctx)
            outs[rank] = (N(s), N(xsy), tuple(out), passes.value)
            L.call("spx_ctx_destroy", ctx)
        except Exception as e:  # pragma: no cover
            errs.append(e)
            barrier.abort()

    th = [threading.Thread(target=worker, args=(k,)) for k in range(world)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errs, errs
    assert outs[0][2] == outs[1][2] and outs[0][3] == outs[1][3]
    s = np.concatenate([o[0] for o in outs])
    ref = N(s_one)
    tol = (64 if dt == np.float64 else 16) * eps(dt) * (np.abs(ref) + np.abs(sj) + 1)
    assert np.all(np.abs(s.astype(np.float64) - ref.astype(np.float64)) <= tol)
    assert bits_equal(np.concatenate([o[1] for o in outs]), ((xk + sj) + s).astype(dt))
    assert float(np.linalg.norm((s + sj).astype(np.float64))) == pytest.approx(delta, rel=1e-10 if dt == np.float64 else 1e-5)
    psi_s, ss, gd = outs[0][2]
    assert psi_s == pytest.approx(res.psi, rel=1e-12 if dt == np.float64 else 1e-5)
    assert math.sqrt(ss) == pytest.approx(res.snorm, rel=1e-10 if dt == np.float64 else 1e-5)
    g64, s64 = grad.astype(np.float64), s.astype(np.float64)
    assert abs(gd - float(np.sum(g64 * s64))) <= 1e-12 * float(np.sum(np.abs(g64 * s64)))


# ------------------------------------------------------------------------------------------------- scale ---
def test_step_l1b2_c3_size():
    """One C3-sized vector (Float32 2^29; Float64 2^27 with SPX_FULLSIZE=0), inputs generated on the device: s bit for
    bit the stand-alone prox!'s, the same pass count, the scalars against torch Float64 sums."""
    from test_gpu_fullsize import dev_uniform

    tdt, n = (torch.float32, 1 << 29) if FULL else (torch.float64, 1 << 27)
    dt = np.float32 if tdt == torch.float32 else np.float64
    xk, sj, g = dev_uniform(n, 0, tdt, 4.0, -2.0), dev_uniform(n, 1, tdt, 1.0, -0.5), dev_uniform(n, 2, tdt, 4.0, -2.0)
    q = g * torch.tensor(dt(-dt(NU)), device=DEV)
    y = torch.empty_like(g)
    p0 = sp.shifted(sp.shifted(sp.NormL1(LAM), xk, 1e30, sp.NormL2(1.0)), sj)
    sp.prox_(y, p0, q, NU)
    delta = 0.5 * float(torch.linalg.vector_norm((sj + y).double()))
    psi = sp.shifted(sp.shifted(sp.NormL1(LAM), xk, delta, sp.NormL2(1.0)), sj)
    sp.prox_(y, psi, q, NU)
    prox_passes = psi.last_passes
    del q
    s, xsy = torch.empty_like(g), torch.empty_like(g)
    _, res = sp.step_(s, psi, g, NU, xsy=xsy)
    assert torch.equal(s, y) and psi.last_passes == prox_passes
    del y
    assert torch.equal(xsy, (xk + sj) + s)
    s64 = s.double()
    assert float(torch.linalg.vector_norm(sj.double() + s64)) == pytest.approx(delta, rel=1e-10 if dt == np.float64 else 1e-5)
    gs = g.double() * s64
    assert res.snorm ** 2 == pytest.approx(float((s64 * s64).sum()), rel=1e-12)
    assert abs(res.gdots - float(gs.sum())) <= 1e-12 * float(gs.abs().sum())
    assert res.psi == pytest.approx(psi(s), rel=1e-12 if dt == np.float64 else 1e-5)
    assert res.psi == pytest.approx(LAM * float((xk.double() + sj.double() + s64).abs().sum()),
                                    rel=1e-12 if dt == np.float64 else 1e-5)
