"""The bulk-copy streaming kernel of the Box operators (ew_bulk_kernel, spx_elementwise.cuh).

Vector bounds at n >= SPX_EWB_MIN_N route ShiftedNormL1Box / ShiftedNormL0Box prox! and ShiftedNormL0Box iprox! through
the producer-warp ring (RootNormLhalfBox and the L1Box iprox! keep ew_kernel; checked here all the same); every output
must be what ew_kernel computes, bit for bit, and what the oracle computes (LhalfBox: tests/gpu_util.py::check_lhalfbox),
at sizes that end on a full tile and on a partial one,
in place, with non-finite and signed-zero operands, both kinds of `selected`, and with the fused ψ(y) equal to
ψ(y) evaluated on its own and the same bits on every run.  The CPU test reads the SASS of the built object."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "shiftedproximaloperators.jl_b200", "csrc")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


def bulk_min_n():
    """SPX_EWB_MIN_N as spx_elementwise.cuh defines it: the smallest n the bulk kernel takes."""
    with open(os.path.join(CSRC, "spx_elementwise.cuh")) as f:
        m = re.search(r"#define SPX_EWB_MIN_N \((\d+) << (\d+)\)", f.read())
    return int(m.group(1)) << int(m.group(2))


NMIN = bulk_min_n()
# the threshold, one past it, a size no tile length divides, and a multiple of every tile length
SIZES = [NMIN, NMIN + 1, NMIN + 333, NMIN + 8192]
DT = [np.float64, np.float32]
SELS = [None, "range", "mask"]


def _cuobjdump(*args):
    return subprocess.run([CUOBJDUMP, *args], capture_output=True, text=True, check=True).stdout


def _functions(text):
    """{kernel name: its part of a cuobjdump listing}"""
    funcs = {}
    for part in re.split(r"\n\s*Function\s*:?\s*", "\n" + text)[1:]:  # "Function : name" (-sass), "Function name:"
        name, _, body = part.partition("\n")
        funcs[name.strip().rstrip(":")] = body
    return funcs


def test_bulk_kernels_use_bulk_copies_and_no_per_thread_async_copies():
    """The instantiations of ew_bulk_kernel that the C2 step runs (L0Box prox! with ψ, L0Box iprox!, Float64) stage their
    operands with cp.async.bulk completing on mbarriers (UBLKCP + SYNCS in their SASS); they live in spx_bulk.o, LhalfBox
    has none, and nothing in spx_elementwise.o uses bulk or per-thread asynchronous copies (UBLKCP, LDGSTS)."""
    ew = os.path.join(CSRC, "build", "spx_elementwise.o")
    bulk = os.path.join(CSRC, "build", "spx_bulk.o")
    if not os.path.exists(CUOBJDUMP):
        pytest.skip("cuobjdump not available")
    if not (os.path.exists(ew) and os.path.exists(bulk)):
        pytest.skip("library not built")
    sass = _cuobjdump("-sass", ew)
    assert "LDGSTS" not in sass and "UBLKCP" not in sass and "ew_bulk_kernel" not in sass
    funcs = _functions(_cuobjdump("-sass", bulk))
    assert not any("ProxLhalfBox" in nm or "IproxL1Box" in nm for nm in funcs)
    for functor in ("9ProxL0BoxIdLb1E", "10IproxL0BoxIdLb0E"):
        bodies = [b for nm, b in funcs.items() if "ew_bulk_kernel" in nm and functor in nm]
        assert len(bodies) == 1, (functor, list(funcs))
        assert "UBLKCP" in bodies[0] and "SYNCS" in bodies[0], functor


def test_elementwise_kernels_reserve_no_shared_memory():
    """A kernel with dynamic shared memory makes nvcc reserve 1 KiB of static shared memory in every kernel of its
    module.  ew_bulk_kernel is kept in spx_bulk.o, so ew_kernel (without a ψ fold: no block reduction) keeps none."""
    ew = os.path.join(CSRC, "build", "spx_elementwise.o")
    if not os.path.exists(CUOBJDUMP):
        pytest.skip("cuobjdump not available")
    if not os.path.exists(ew):
        pytest.skip("library not built")
    funcs = _functions(_cuobjdump("-res-usage", ew))
    lhalf = [b for nm, b in funcs.items() if nm.startswith("_ZN3spx9ew_kernel") and "ProxLhalfBoxIdLb0E" in nm]
    assert lhalf and all("SHARED:0 " in b for b in lhalf), lhalf


# ------------------------------------------------------------------------------------------------------------- GPU --
def _gpu():
    from gpu_util import DEV, N, T, bounds, check_lhalfbox, diag, inputs, orc, sp
    return DEV, N, T, bounds, check_lhalfbox, diag, inputs, orc, sp


def _plant(a, vals, k):
    """non-finite / signed-zero entries in operand k: spread over the tiles, and in the last elements (the tail)"""
    n = a.size
    pos = (np.arange(64, dtype=np.int64) * 104_729 + k * 7_919) % n
    a[pos] = np.resize(np.asarray(vals, a.dtype), pos.size)
    a[n - 1 - k] = a.dtype.type(vals[k % len(vals)])
    return a


def _operands(n, dt, special=True):
    _, _, _, bounds, _, diag, inputs, _, _ = _gpu()
    xk, sj, q = inputs(n, dt)
    l, u = bounds(n, dt)
    d = diag(n, dt)
    if not special:
        return xk, sj, q, l, u, d
    sp_all = [np.nan, np.inf, -np.inf, 0.0, -0.0]
    for k, a in enumerate((xk, sj, q)):
        _plant(a, sp_all, k)
    _plant(l, [np.nan, -np.inf, 0.0, -0.0], 3)  # keeps l <= u wherever both are numbers
    _plant(u, [np.nan, np.inf, -0.0, 0.0], 4)
    eps = np.finfo(dt).eps
    _plant(d, [np.nan, np.inf, -np.inf, 0.0, -0.0, eps, -eps, eps / 2, -eps / 2, -1e-30, 1e-30, -2.0], 5)
    return xk, sj, q, l, u, d


def _sel(kind, n):
    if kind is None:
        return None, None
    if kind == "range":
        return range(1, n, 3), np.arange(1, n, 3)
    lst = np.random.default_rng(11).integers(0, n, size=n // 2)
    return lst.tolist(), lst


def _off(T, a):
    """a on the device one element past a 16-byte boundary: the same values through ew_kernel"""
    return T(np.concatenate([a[:1], a]))[1:]


def _psi_rel(name, dt):
    """fused ψ(y) against ψ(y) evaluated on its own (test_gpu_parity.py::test_box_values): the L0 count exactly, the
    other sums to 1e-12 (Float64) / 2e-6 (Float32: the terms are formed in Float32, summed in a different order)"""
    return 0.0 if name == "l0" else (1e-12 if dt == np.float64 else 2e-6)


def _check_psi(name, dt, selk, v, v_ew, v_alone):
    """the fused ψ(y) of the bulk kernel against ew_kernel's fused ψ(y) and against ψ(y) on its own (not for a MASK from a
    list with duplicates: the fused sum is over the set, ψ(y) over the list; test_gpu_parity.py::test_box_values)"""
    rel = _psi_rel(name, dt)
    assert _same_scalar(v, v_ew, rel), (name, v, v_ew)
    if selk != "mask":
        assert _same_scalar(v, v_alone, rel), (name, v, v_alone)


def _same_scalar(a, b, rel):
    if np.isnan(a) or np.isnan(b):
        return np.isnan(a) and np.isnan(b)
    if np.isinf(a) or np.isinf(b) or rel == 0:
        return a == b
    return abs(a - b) <= rel * max(1.0, abs(b))


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("selk", SELS)
@pytest.mark.parametrize("special", [False, True])
def test_bulk_box_prox(dt, n, selk, special):
    DEV, N, T, _, check_lhalfbox, _, _, orc, sp = _gpu()
    xk, sj, q, l, u, _ = _operands(n, dt, special)
    sel_dev, sel_host = _sel(selk, n)
    lam, sigma = 1.0, 0.1
    for name, h in (("l1", sp.NormL1(lam)), ("l0", sp.NormL0(lam)), ("lhalf", sp.RootNormLhalf(lam))):
        psi = sp.shifted(sp.shifted(h, T(xk), T(l), T(u), sel_dev), T(sj))
        y = torch.empty(n, dtype=T(q).dtype, device=DEV)
        _, v = sp.prox_(y, psi, T(q), sigma, want_value=True)
        got = N(y)
        if name != "lhalf":
            ref = orc.prox_box(name, xk, sj, q, l, u, lam, sigma, selected=sel_host)
            assert np.array_equal(got, ref, equal_nan=True), (name, np.flatnonzero(got != ref)[:5])
        elif not special:
            check_lhalfbox(got, xk, sj, q, l, u, lam, sigma, selected=sel_host, label=f"bulk {dt.__name__} n={n}")
        # the same bits as ew_kernel (operands off the 16-byte grid), non-finite operands included
        psi_ew = sp.shifted(sp.shifted(h, _off(T, xk), _off(T, l), _off(T, u), sel_dev), _off(T, sj))
        y_ew = _off(T, np.zeros(n, dt))
        _, v_ew = sp.prox_(y_ew, psi_ew, _off(T, q), sigma, want_value=True)
        assert np.array_equal(got.view(np.uint8), N(y_ew).view(np.uint8)), name
        _check_psi(name, dt, selk, v, v_ew, psi(y))
        # a second run: same y bits, same ψ bits (one partial per CTA, folded in a fixed order)
        y2 = torch.empty_like(y)
        _, v2 = sp.prox_(y2, psi, T(q), sigma, want_value=True)
        assert torch.equal(y.view(torch.int64 if dt == np.float64 else torch.int32),
                           y2.view(torch.int64 if dt == np.float64 else torch.int32)), name
        assert np.asarray(v).tobytes() == np.asarray(v2).tobytes(), (name, v, v2)
        # in place: y aliasing q
        yq = T(q).clone()
        sp.prox_(yq, psi, yq, sigma)
        assert np.array_equal(N(yq), got, equal_nan=True), name


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("selk", SELS)
@pytest.mark.parametrize("special", [False, True])
def test_bulk_box_iprox(dt, n, selk, special):
    DEV, N, T, _, _, _, _, orc, sp = _gpu()
    xk, sj, g, l, u, d = _operands(n, dt, special)
    sel_dev, sel_host = _sel(selk, n)
    lam = 0.8
    for name, h in (("l1", sp.NormL1(lam)), ("l0", sp.NormL0(lam))):
        psi = sp.shifted(sp.shifted(h, T(xk), T(l), T(u), sel_dev), T(sj))
        y = torch.empty(n, dtype=T(g).dtype, device=DEV)
        _, v = sp.iprox_(y, psi, T(g), T(d), want_value=True)
        got = N(y)
        # the same bits as ew_kernel (operands off the 16-byte grid)
        psi_ew = sp.shifted(sp.shifted(h, _off(T, xk), _off(T, l), _off(T, u), sel_dev), _off(T, sj))
        y_ew = _off(T, np.zeros(n, dt))
        _, v_ew = sp.iprox_(y_ew, psi_ew, _off(T, g), _off(T, d), want_value=True)
        assert np.array_equal(got.view(np.uint8), N(y_ew).view(np.uint8)), name
        ref = orc.iprox_box(name, xk, sj, g, d, l, u, lam, selected=sel_host)
        keep = np.ones(n, bool)
        if name == "l0":  # IproxL0Box's straight-line selects and the reference's branches part on NaN operands, in
            # ew_kernel as well (bit-identical above): not this kernel's business
            keep = ~(np.isnan(xk) | np.isnan(sj) | np.isnan(g) | np.isnan(d) | np.isnan(l) | np.isnan(u))
        assert np.array_equal(got[keep], ref[keep], equal_nan=True), (name, np.flatnonzero(got[keep] != ref[keep])[:5])
        _check_psi(name, dt, selk, v, v_ew, psi(y))
        _, v2 = sp.iprox_(torch.empty_like(y), psi, T(g), T(d), want_value=True)
        assert np.asarray(v).tobytes() == np.asarray(v2).tobytes(), (name, v, v2)
        # in place: y aliasing g
        yg = T(g).clone()
        sp.iprox_(yg, psi, yg, T(d))
        assert np.array_equal(N(yg), got, equal_nan=True), name


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@pytest.mark.gpu
def test_bulk_routing():
    """Vector bounds at n >= SPX_EWB_MIN_N take ew_bulk_kernel; one element less, scalar bounds, or an operand that is
    not 16-byte aligned keep ew_kernel."""
    DEV, N, T, _, _, _, _, orc, sp = _gpu()
    n = NMIN + 1
    xk, sj, q, l, u, _ = _operands(n, np.float64)
    txk, tsj, tq, tl, tu = map(T, (xk, sj, q, l, u))
    y = torch.empty(n, dtype=torch.float64, device=DEV)

    def run(m, lb, ub, off=0):
        psi = sp.shifted(sp.shifted(sp.NormL0(1.0), txk[off:off + m], lb, ub), tsj[off:off + m])
        return _kernels(lambda: sp.prox_(y[off:off + m], psi, tq[off:off + m], 0.1))

    names = run(NMIN, tl[:NMIN], tu[:NMIN])
    assert any("ew_bulk_kernel" in s for s in names), names
    for names in (run(NMIN - 1, tl[:NMIN - 1], tu[:NMIN - 1]), run(NMIN, -1.0, 1.0),
                  run(NMIN, tl[1:NMIN + 1], tu[1:NMIN + 1], off=1)):
        assert not any("ew_bulk_kernel" in s for s in names) and any("ew_kernel" in s for s in names), names
