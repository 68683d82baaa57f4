"""CPU-side checks of the drop-in boundary (no compute calls): the C-ABI library is built, loads,
and exports every symbol include/shiftedprox.h declares; the host mirror imports without a GPU and
refuses to compute without one (no CPU fallback)."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "shiftedprox.h")
LIB = os.path.join(ROOT, "shiftedproximaloperators.jl_b200", "libshiftedprox.so")
# the toolkit's bin directory need not be on PATH: the build itself calls nvcc by this location (csrc/Makefile)
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


def declared_symbols():
    pre = subprocess.run(["gcc", "-E", "-P", HEADER], check=True, capture_output=True, text=True).stdout
    names = set(re.findall(r"\b(spx_[a-z0-9_]+)\s*\(", pre))
    names -= {"spx_allreduce_sum_fn"}
    return sorted(names)


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(LIB):
        import __graft_entry__ as g

        g.build()
    return ctypes.CDLL(LIB)


def test_header_compiles_as_c():
    subprocess.run(["gcc", "-std=c99", "-fsyntax-only", "-x", "c", HEADER], check=True)


def test_library_exports_every_declared_symbol(lib):
    names = declared_symbols()
    assert len(names) >= 70, names
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    for suf in ("f64", "f32"):
        for op in ("prox_l1", "iprox_l1", "prox_l0", "iprox_l0", "prox_lhalf", "prox_l1box", "iprox_l1box",
                   "prox_l0box", "iprox_l0box", "prox_lhalfbox", "prox_l1b2", "prox_l1b2_sharded", "prox_groupl2",
                   "prox_groupl2binf", "prox_indballl0", "value_sep", "value_box", "value_l1b2", "value_binf",
                   "value_groupl2", "value_partial", "box_host", "box_multi_host", "prox_indballl0_sharded", "step_sep",
                   "step_box"):
            assert f"spx_{op}_{suf}" in names


def test_version_and_scalar_helpers(lib):
    assert lib.spx_version() >= 100
    lib.spx_prox_zero_f64.restype = ctypes.c_double
    lib.spx_iprox_zero_f64.restype = ctypes.c_double
    d = ctypes.c_double
    # prox_zero / iprox_zero are plain host functions (ShiftedProximalOperators.jl:203, :217-236)
    assert lib.spx_prox_zero_f64(d(5.0), d(-1.0), d(2.0)) == 2.0
    assert lib.spx_iprox_zero_f64(d(2.0), d(1.0), d(-1.0), d(2.0)) == -0.5
    assert lib.spx_iprox_zero_f64(d(-2.0), d(1.0), d(-1.0), d(2.0)) == 2.0
    assert lib.spx_iprox_zero_f64(d(0.0), d(2.0), d(-1.0), d(1.0)) == -1.0
    assert lib.spx_iprox_zero_f64(d(0.0), d(0.0), d(-1.0), d(1.0)) == 0.0


def test_library_is_sm100a_only():
    out = subprocess.run([CUOBJDUMP, "--list-elf", LIB], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_host_mirror_imports_and_fails_loudly_without_gpu():
    import torch

    import shiftedprox as sp

    h = sp.NormL1(1.0)
    assert h.lam == 1.0
    with pytest.raises(ValueError):
        sp.IndBallL0(0)
    if not torch.cuda.is_available():
        with pytest.raises(TypeError):
            sp.shifted(h, torch.ones(4, dtype=torch.float64))  # host tensor: no CPU path
        with pytest.raises(RuntimeError):
            sp.context(0)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "shiftedproximaloperators.jl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".jl")):
                text = open(os.path.join(dirpath, f), encoding="utf-8").read()
                assert "liboracle" not in text and "from oracle" not in text and "import oracle" not in text, f


def test_group_index_sets_must_be_contiguous_ranges():
    """The reference's GroupNormL2 accepts any index collection per group (groupNormL2.jl:15-31); the device layout is
    CSR offsets, so the host layer rejects anything that is not a partition of the vector into contiguous ranges in
    order -- at construction, loudly (documented in DESIGN.md §7 and include/shiftedprox.h)."""
    import pytest
    import shiftedprox as sp

    sp.GroupNormL2([1.0, 2.0], [range(0, 3), range(3, 6)])  # fine
    with pytest.raises(ValueError, match="contiguous ranges"):
        sp.GroupNormL2([1.0, 2.0], [range(0, 3), range(4, 6)])  # gap
    with pytest.raises(ValueError, match="contiguous ranges"):
        sp.GroupNormL2([1.0, 2.0], [range(3, 6), range(0, 3)])  # out of order
    with pytest.raises(ValueError, match="same"):
        sp.GroupNormL2([1.0], [range(0, 3), range(3, 6)])


def test_library_holds_only_sm_100a_code_and_the_bulk_copy_kernels_use_tma():
    """The shipped library is sm_100a-only (no PTX fallback, no other architecture), and the CTA-per-group kernels of
    spx_group.cu stage their groups with bulk copies (UBLKCP in the SASS: cp.async.bulk completing on an mbarrier) --
    checked on the built artefacts with cuobjdump (skipped when the toolkit has none)."""
    if not os.path.exists(CUOBJDUMP):
        pytest.skip("cuobjdump not available")
    pkg = os.path.join(ROOT, "shiftedproximaloperators.jl_b200")
    elfs = subprocess.run([CUOBJDUMP, "-lelf", os.path.join(pkg, "libshiftedprox.so")], capture_output=True, text=True).stdout
    names = [ln.split(":")[-1].strip() for ln in elfs.splitlines() if "ELF file" in ln]
    assert names and all(n.endswith(".sm_100a.cubin") for n in names), names
    ptx = subprocess.run([CUOBJDUMP, "-lptx", os.path.join(pkg, "libshiftedprox.so")], capture_output=True, text=True).stdout
    assert "PTX file" not in ptx
    obj = os.path.join(pkg, "csrc", "build", "spx_group.o")
    if os.path.exists(obj):
        sass = subprocess.run([CUOBJDUMP, "-sass", obj], capture_output=True, text=True).stdout
        assert sass.count("UBLKCP") > 0 and "SYNCS" in sass  # bulk copy + mbarrier
