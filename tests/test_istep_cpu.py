"""CPU checks of the fused step around iprox! (spx_istep_sep_* / spx_istep_box_*): the library exports it for both
element types, the oracle's composition (istep_oracle.solver_istep) agrees with a numpy restatement of iprox! and the
sums, and no istep instance of step_kernel touches local memory."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from istep_oracle import solver_istep
from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "shiftedproximaloperators.jl_b200")
LIB = os.path.join(PKG, "libshiftedprox.so")
STEP_O = os.path.join(PKG, "csrc", "build", "spx_step.o")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


def _built():
    if not (os.path.exists(LIB) and os.path.exists(STEP_O)):
        import __graft_entry__ as g

        g.build()


def test_istep_symbols_are_exported():
    _built()
    lib = ctypes.CDLL(LIB)
    for name in ("spx_istep_sep", "spx_istep_box"):
        for suf in ("f64", "f32"):
            assert hasattr(lib, f"{name}_{suf}"), f"{name}_{suf}"


def _numpy_iprox(op, xk, sj, g, d, lam):
    """shiftedNormL1.jl:60-75 / shiftedNormL0.jl:61-80, element by element in the vectors' type"""
    dt = g.dtype.type
    lam = dt(lam)
    if op == "l1":
        t = (-xk) - sj
        c = (-g) / d
        w = lam / d
        return np.minimum(np.maximum(t, c - w), c + w)
    xps = xk + sj
    ci = np.sqrt(dt(2) * lam * d)
    return np.where(np.abs(d * xps - g) <= ci, -xps, (-g) / d)


def _inputs(n, dt):
    xk = orc.uniform(n, 0, dt, 4.0, -2.0)
    sj = orc.uniform(n, 1, dt, 1.0, -0.5)
    g = orc.uniform(n, 2, dt, 4.0, -2.0)
    D = orc.uniform(n, 5, dt, 1.0, 0.5)
    return xk, sj, g, D


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("op", ["l1", "l0"])
@pytest.mark.parametrize("dshift", [0.0, 0.25])
def test_solver_istep_matches_numpy(dt, op, dshift):
    n = 1237
    xk, sj, g, D = _inputs(n, dt)
    lam = 0.9
    s, xsy, psi, snorm, gdots, sds = solver_istep(op, xk, sj, g, D, dshift, lam)
    d = D + dt(dshift)
    assert d.dtype == dt
    ref = _numpy_iprox(op, xk, sj, g, d, lam)
    assert np.array_equal(s, ref)
    assert np.array_equal(xsy, (xk + sj) + ref)
    v = (xk + sj) + ref
    h = np.sum(np.abs(v.astype(np.float64))) if op == "l1" else float(np.count_nonzero(v))
    assert psi == pytest.approx(float(dt(lam) * dt(h)), rel=1e-12 if dt == np.float64 else 1e-6)
    s64, g64, d64 = ref.astype(np.float64), g.astype(np.float64), d.astype(np.float64)
    assert snorm == pytest.approx(np.sqrt(np.sum(s64 * s64)), rel=1e-14)
    assert gdots == pytest.approx(np.sum(g64 * s64), rel=1e-12)
    assert sds == pytest.approx(np.sum(d64 * s64 * s64), rel=1e-12)


def test_solver_istep_hand_computed_l1():
    xk = np.array([1.0, -2.0, 0.5]); sj = np.zeros(3); g = np.array([1.0, 1.0, -4.0]); D = np.array([1.0, 0.5, 1.5])
    s, xsy, psi, snorm, gdots, sds = solver_istep("l1", xk, sj, g, D, 0.5, 1.0)
    # d = [1.5, 1, 2];  s = min(max(-xk, -g/d - λ/d), -g/d + λ/d)   (shiftedNormL1.jl:60-75)
    assert np.array_equal(s, [-1.0, 0.0, 1.5])
    assert np.array_equal(xsy, [0.0, -2.0, 2.0])
    assert psi == 4.0 and snorm == pytest.approx(np.sqrt(3.25)) and gdots == -7.0
    assert sds == 1.5 * 1.0 + 1.0 * 0.0 + 2.0 * 2.25


def test_solver_istep_asserts_on_shifted_d():
    xk, sj, g, D = _inputs(64, np.float64)
    D[17] = -0.1
    with pytest.raises(AssertionError, match=r"d\[17\]"):
        solver_istep("l0", xk, sj, g, D, 0.0, 1.0)
    solver_istep("l0", xk, sj, g, D, 0.25, 1.0)  # every D + σ > 0


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("op", ["l1", "l0"])
def test_solver_istep_box_is_iprox_plus_value(dt, op):
    n = 1237
    xk, sj, g, D = _inputs(n, dt)
    D = np.where(np.arange(n) % 10 == 3, -D, D).astype(dt)
    l = -(dt(0.25) + orc.uniform(n, 3, dt)); u = dt(0.25) + orc.uniform(n, 4, dt)
    sel = np.arange(0, n, 2)
    s, xsy, psi, _, _, sds = solver_istep(op, xk, sj, g, D, 0.25, 0.8, l, u, sel)
    d = D + dt(0.25)
    ref = orc.iprox_box(op, xk, sj, g, d, l, u, 0.8, sel)
    assert np.array_equal(s, ref) and psi == orc.value_box(op, xk, sj, ref, l, u, 0.8, sel)
    s64 = ref.astype(np.float64)
    assert sds == pytest.approx(np.sum(d.astype(np.float64) * s64 * s64), rel=1e-12)


def _functions(text):
    funcs = {}
    for part in re.split(r"\n\s*Function\s*:\s*", "\n" + text)[1:]:
        name, _, body = part.partition("\n")
        funcs[name.strip()] = body
    return funcs


def test_istep_kernels_use_no_local_memory():
    """Every istep instance of step_kernel (the ones on an Iprox functor) keeps its operands and sums in registers: no
    LDL / STL in its SASS."""
    _built()
    if not os.path.exists(CUOBJDUMP):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([CUOBJDUMP, "-sass", STEP_O], capture_output=True, text=True, check=True).stdout
    funcs = {k: v for k, v in _functions(sass).items() if "step_kernel" in k and "Iprox" in k}
    assert len(funcs) == 16, sorted(funcs)  # {L1, L0, L1Box, L0Box} x {f64, f32} x {vector, scalar}
    for name, body in funcs.items():
        assert not re.search(r"\b(LDL|STL)\b", body), name
