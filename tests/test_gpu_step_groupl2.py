"""GPU tests of the ShiftedGroupNormL2 solver step (spx_step_groupl2_*) on every group layout.

The step runs in the passes of the prox! kernels of the layout's group sizes: the packed warp rounds (<= 256 elements),
the CTA-per-group classes (257..1024 and 1025..4096), the warp path of longer groups, and the two grid-wide passes of a
single group spanning the vector.  Bars, in both precisions:
  - s bit for bit the stand-alone prox! of q = fl(-ν∇f), xsy bit for bit (xk + sj) + s;
  - ψ(s) against the oracle's value at the GPU's s and against ψ(s) of the library, Σs² and Σ∇f·s against Float64 sums
    of the GPU's own s;
  - two identical calls give identical scalars, with and without xsy; x <- x + s (xsy = xk) is accepted;
  - fewer launches than the composed form (ShiftedProximableFunction.step_), and no step_pre / step_post kernel;
  - a layout rewritten after validation (stale census) or never validated is still computed correctly.
"""
import numpy as np
import pytest
import torch

from gpu_util import DEV, N, T, inputs, orc, sp
from test_gpu_step import scalars_close
from test_gpu_step_scale import group_windows, launches, same_scalars

pytestmark = pytest.mark.gpu

DT = [np.float64, np.float32]
NU = 0.3


def sizes_of(layout):
    rng = np.random.default_rng(11)
    if layout == "ragged":  # 1..4096, log-uniform: every size class
        return np.floor(np.exp(rng.uniform(0, np.log(4097), 700))).astype(np.int64).clip(1, 4096)
    if layout == "edges":  # both sides of every class boundary
        return np.tile([1024, 1025, 4096, 4097, 256, 257, 1, 8, 9, 64, 65, 512, 513, 2048, 2049], 6)
    if layout == "long":  # groups of the warp path only
        return np.array([5000, 70000, 3, 300, 5000, 1, 70000])
    if layout == "mid":  # the 128-thread class only
        return rng.integers(257, 1025, 300)
    if layout == "two":
        return np.array([777, 100_003])
    raise ValueError(layout)


def offsets_of(sizes):
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)


def problem(dt, sizes, unaligned=False):
    offs = offsets_of(sizes)
    n = int(offs[-1])
    k = 1 if unaligned else 0  # views one element into their buffers: the bulk copies' front padding
    xk, sj, grad = inputs(n + k, dt)
    xk, sj, grad = xk[k:], sj[k:], grad[k:]
    txk, tsj, tg = (T(np.concatenate([np.zeros(k, dt), a]))[k:] for a in (xk, sj, grad))
    lam_g = (dt(0.5) + orc.uniform(len(sizes), 12, dt)).astype(dt)
    psi = sp.shifted(sp.shifted(sp.GroupNormL2(T(lam_g), None, offsets=T(offs)), txk), tsj)
    return offs, xk, sj, grad, tg, lam_g, psi


def empty_like(t, unaligned):
    k = 1 if unaligned else 0
    return torch.empty(t.numel() + k, dtype=t.dtype, device=DEV)[k:]


def prox_ref(psi, grad, dt, like):
    y = torch.empty_like(like)
    sp.prox_(y, psi, T((dt(-dt(NU)) * grad).astype(dt)), NU)
    return y


def check_result(res, s, xsy, xk, sj, grad, offs, lam_g, psi, dt):
    gs = N(s)
    if xsy is not None:
        assert np.array_equal(N(xsy), ((xk + sj) + gs).astype(dt))
    g64, s64 = grad.astype(np.float64), gs.astype(np.float64)
    scalars_close(res, orc.value_groupl2(xk, sj, gs, offs, lam_g), float(np.sqrt(np.sum(s64 * s64))),
                  float(np.sum(g64 * s64)), grad, gs, dt)
    assert res.psi == pytest.approx(psi(s), rel=1e-12 if dt == np.float64 else 1e-6, abs=1e-300)


def kernel_names(fn):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("layout", ["ragged", "edges", "long", "mid", "two"])
@pytest.mark.parametrize("unaligned", [False, True])
def test_step_groupl2_every_layout(dt, layout, unaligned):
    offs, xk, sj, grad, tg, lam_g, psi = problem(dt, sizes_of(layout), unaligned)
    s, xsy = empty_like(tg, unaligned), empty_like(tg, unaligned)
    (_, res), nl = launches(lambda: sp.step_(s, psi, tg, NU, xsy=xsy))
    assert torch.equal(s, prox_ref(psi, grad, dt, s))
    check_result(res, s, xsy, xk, sj, grad, offs, lam_g, psi, dt)
    # deterministic sums, with and without xsy
    s2 = empty_like(tg, unaligned)
    _, res2 = sp.step_(s2, psi, tg, NU)
    assert torch.equal(s2, s) and same_scalars(res2, res)
    _, res3 = sp.step_(s2, psi, tg, NU, xsy=xsy)
    assert same_scalars(res3, res)
    # fewer launches than the composed form, none of them step_pre / step_post
    s_c, xsy_c = torch.empty_like(s), torch.empty_like(s)
    (_, res_c), nl_c = launches(lambda: sp.ShiftedProximableFunction.step_(psi, s_c, tg, NU, xsy=xsy_c))
    assert torch.equal(s_c, s) and torch.equal(xsy_c, xsy)
    assert nl < nl_c, (nl, nl_c)
    names = kernel_names(lambda: sp.step_(s2, psi, tg, NU, xsy=xsy))
    assert names and not any("StepPre" in k or "StepPost" in k for k in names), names


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("layout", ["ragged", "two"])
def test_step_groupl2_in_place_and_alias_rules(dt, layout):
    offs, xk, sj, grad, tg, lam_g, psi = problem(dt, sizes_of(layout))
    s = torch.empty_like(tg)
    y = prox_ref(psi, grad, dt, s)
    _, res = sp.step_(s, psi, tg, NU)  # xsy = None
    assert torch.equal(s, y)
    check_result(res, s, None, xk, sj, grad, offs, lam_g, psi, dt)
    # x <- x + s: xsy is ψ's own xk
    s2 = torch.empty_like(s)
    _, res2 = sp.step_(s2, psi, tg, NU, xsy=psi.xk)
    assert torch.equal(s2, y) and same_scalars(res2, res)
    assert np.array_equal(N(psi.xk), ((xk + sj) + N(s2)).astype(dt))
    # refused, as before: s on ∇f, s on xk, partial overlaps
    n = tg.numel()
    with pytest.raises(ValueError):
        sp.step_(tg, psi, tg, NU)
    with pytest.raises(ValueError):
        sp.step_(psi.xk, psi, tg, NU)
    buf = T(np.concatenate([grad, grad]))
    with pytest.raises(ValueError):
        sp.step_(buf[1:n + 1], psi, buf[:n], NU)
    with pytest.raises(ValueError):
        sp.step_(s2, psi, buf[:n], NU, xsy=buf[1:n + 1])


@pytest.mark.parametrize("dt", DT)
def test_step_groupl2_stale_census_gains_long_groups_with_xsy_on_xk(dt):
    """A layout validated with groups of <= 256 elements, rewritten in place to hold a mid, a big and a > 4096 group:
    the packed kernel flags them, the long-group kernels take only those, and x <- x + s is still right."""
    rng = np.random.default_rng(5)
    sizes = rng.integers(1, 257, 400)
    offs, xk, sj, grad, tg, lam_g, psi = problem(dt, sizes)
    new = sizes.copy()
    new[10] += 700  # 257..1024
    new[100] += 3000  # 1025..4096
    new[200] += 6000  # > 4096
    new[300] = 1
    left = int(new.sum() - sizes.sum())
    j = 399
    while left > 0:  # keep n: take the surplus from the tail (groups may become empty)
        t = min(left, int(new[j]))
        new[j] -= t
        left -= t
        j -= 1
    offs2 = offsets_of(new)
    assert offs2[-1] == offs[-1] and sorted(np.diff(offs2))[-3:][0] > 256
    psi._offs.copy_(T(offs2))
    s = torch.empty_like(tg)
    y = prox_ref(psi, grad, dt, s)
    (_, res), nl = launches(lambda: sp.step_(s, psi, tg, NU, xsy=psi.xk))
    assert torch.equal(s, y)
    assert np.array_equal(N(psi.xk), ((xk + sj) + N(s)).astype(dt))
    g64, s64 = grad.astype(np.float64), N(s).astype(np.float64)
    scalars_close(res, orc.value_groupl2(xk, sj, N(s), offs2, lam_g), float(np.sqrt(np.sum(s64 * s64))),
                  float(np.sum(g64 * s64)), grad, N(s), dt)


@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("how", ["loses_classes", "never_validated"])
def test_step_groupl2_census_stale_or_missing(dt, how):
    sizes = np.ones(3000, np.int64)
    sizes[::500] = 600
    sizes[250::1000] = 3000
    sizes[777] = 5000
    offs, xk, sj, grad, tg, lam_g, psi = problem(dt, sizes)
    if how == "loses_classes":  # validated with every class, rewritten to groups of <= 256
        n, ng = int(offs[-1]), len(offs) - 1
        offs2 = np.round(np.linspace(0, n, ng + 1)).astype(np.int64)
        assert np.diff(offs2).max() <= 256
        psi._offs.copy_(T(offs2))
    else:  # the same layout in a buffer spx_group_validate_offsets never saw
        offs2 = offs
        psi._offs = T(offs).clone()
    s, xsy = torch.empty_like(tg), torch.empty_like(tg)
    _, res = sp.step_(s, psi, tg, NU, xsy=xsy)
    assert torch.equal(s, prox_ref(psi, grad, dt, s))
    check_result(res, s, xsy, xk, sj, grad, offs2, lam_g, psi, dt)
    _, again = sp.step_(s, psi, tg, NU, xsy=xsy)
    assert same_scalars(again, res)


@pytest.mark.parametrize("dt", DT)
def test_step_groupl2_every_persistent_grid_loops(dt):
    """About 1.2 million groups, mostly of two elements, with every class sprinkled over the whole layout: every
    persistent grid of the step walks >= 3 chunks.  Windows of whole groups against the oracle at 8 ulp of the value
    scale, s against prox!, the sums against Float64 sums of the GPU's s."""
    ng = 1_200_000
    sizes = np.full(ng, 2, np.int64)
    sizes[::997] = 300
    sizes[::2999] = 2000
    sizes[::20011] = 5000
    offs, xk, sj, grad, tg, lam_g, psi = problem(dt, sizes)
    s, xsy = torch.empty_like(tg), torch.empty_like(tg)
    _, res = sp.step_(s, psi, tg, NU, xsy=xsy)
    assert torch.equal(s, prox_ref(psi, grad, dt, s))
    gs = N(s)
    assert np.array_equal(N(xsy), ((xk + sj) + gs).astype(dt))
    g64, s64 = grad.astype(np.float64), gs.astype(np.float64)
    # ψ: the oracle sums its 1.2e6 terms in R, which in Float32 drifts by more than the bar; the reference here is
    # λ_g ‖v_g‖ of the GPU's s rounded to R per group (v = (xk + sj) + s in R), the terms summed in Float64
    v = ((xk + sj) + gs).astype(np.float64)
    terms = (lam_g * np.sqrt(np.add.reduceat(v * v, offs[:-1])).astype(dt)).astype(np.float64)
    ref_psi = float(dt(terms.sum())) if dt == np.float32 else orc.value_groupl2(xk, sj, gs, offs, lam_g)
    scalars_close(res, ref_psi, float(np.sqrt(np.sum(s64 * s64))), float(np.sum(g64 * s64)), grad, gs, dt)
    _, again = sp.step_(s, psi, tg, NU, xsy=xsy)
    assert same_scalars(again, res)
    q = (dt(-dt(NU)) * grad).astype(dt)
    eps = np.finfo(dt).eps
    rng = np.random.default_rng(3)
    wg = 30_000
    for g0 in group_windows(ng, wg, rng):
        a, b = int(offs[g0]), int(offs[g0 + wg])
        ref = orc.prox_groupl2(xk[a:b], sj[a:b], q[a:b], offs[g0:g0 + wg + 1] - a, lam_g[g0:g0 + wg], NU)
        scale = np.abs(xk[a:b]).astype(np.float64) + np.abs(sj[a:b]) + np.abs(q[a:b]) + 1
        assert np.all(np.abs(gs[a:b].astype(np.float64) - ref) <= 8 * eps * scale), g0


@pytest.mark.parametrize("dt", DT)
def test_step_groupl2_single_group_from_norml2(dt):
    """ShiftedGroupNormL2 built from NormL2 (one group spanning the vector): norm pass and scaling pass, aligned and
    one element off, against prox! and the oracle."""
    for unaligned in (False, True):
        n = 1 << 20
        k = 1 if unaligned else 0
        xk, sj, grad = inputs(n + k, dt)
        txk, tsj, tg = T(xk)[k:], T(sj)[k:], T(grad)[k:]
        xk, sj, grad = xk[k:], sj[k:], grad[k:]
        psi = sp.shifted(sp.shifted(sp.NormL2(0.7), txk), tsj)
        s, xsy = empty_like(tg, unaligned), empty_like(tg, unaligned)
        (_, res), nl = launches(lambda: sp.step_(s, psi, tg, NU, xsy=xsy))
        assert torch.equal(s, prox_ref(psi, grad, dt, s))
        check_result(res, s, xsy, xk, sj, grad, np.array([0, n]), np.array([0.7], dt), psi, dt)
        _, again = sp.step_(s, psi, tg, NU)
        assert same_scalars(again, res)
        (_, _), nl_c = launches(lambda: sp.ShiftedProximableFunction.step_(psi, torch.empty_like(s), tg, NU))
        assert nl < nl_c
