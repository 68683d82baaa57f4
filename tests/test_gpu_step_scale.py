"""The fused solver steps at the sizes where their kernels loop, against the oracle.

Every step kernel is persistent: a block, warp or CTA walks several tiles, rounds or problems and carries the step's
sums (ψ(s), Σs², Σ∇f·s, Σd s²) from one to the next.  The sizes here are worked out from the bounds in the sources
(2048 resident threads per SM, kMaxPartials, the tile lengths, the top-r instance thresholds), parsed from csrc/ so that
a retune fails test_step_scale_constants_match_the_sources instead of quietly shrinking the coverage, and each test
asserts the loop condition it relies on.

  A. step_kernel (spx_step_sep / spx_step_box / spx_istep_sep / spx_istep_box): every block runs >= 3 tiles and the
     last one the scalar tail.
  B. the top-r step (spx_step_indballl0) on each of the four topr_stream_kernel instances, every CTA walking >= 3
     problems, with hard problems spread over the grid for the radix and fixup kernels.
  C. the uniform-layout GroupNormL2Binf step with >= 3 rounds per warp, and the one-pass GroupNormL2 step.
  D. the BASELINE.json shapes end to end (C1, the C2 operands, C4, C5) and an element index past 2^31.
     SPX_FULLSIZE=0 runs section D at 1/64 of the size (never below what its loop conditions need).

Bars: s bit-identical to the oracle for the exact operators (RootNormLhalf(Box): the bars of test_prox_lhalf /
check_lhalfbox; the group types: check_groupl2binf or 8 ulp of the value scale) and to the stand-alone prox!/iprox! on
the device over the whole vector; xsy bit-identical to (xk + sj) + s; ψ(s) exact for the L0 and top-r counts, else to
1e-12 / 1e-5 (Float64 / Float32); Σs² to 1e-12 relative, Σ∇f·s and Σd s² to 1e-12 of their sums of magnitudes, against
Float64 sums; three identical calls give the same scalars bit for bit; the route (launch count, kernel instance) is
the one the test means to exercise.  Two bars differ from the small-size tests, both because of the reference side: the
Float32 ψ of GroupNormL2Binf is compared with a Float64 sum of its terms (the oracle sums ψ in R, and over 2^23
elements its own rounding reaches 1e-5), and the groups planted with |∇f| ~ 1e13 are pinned to prox! bit for bit but
left out of the oracle windows (their s is the difference of two ~1e12 magnitudes, which neither the support nor 8 ulp
of the scale can pin down; their neighbours in the same declined rounds are checked).
"""
import math
import os
import re
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

from gpu_util import DEV, N, T, bounds, check_groupl2binf, check_lhalfbox, diag, inputs, orc, sp
from istep_oracle import solver_istep
from test_gpu_fullsize import c2_host_inputs, dev_checksum, dev_uniform, host_checksum

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "shiftedproximaloperators.jl_b200", "csrc")

FULL = os.environ.get("SPX_FULLSIZE", "1") != "0"
SHRINK = 0 if FULL else 6
DT = [np.float64, np.float32]
THREADS_PER_SM = 2048  # resident threads per SM of sm_100: the bound of every persistent grid below
gpu = pytest.mark.gpu


# ---------------------------------------------------------------- constants of the sources ---
def _source(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _const(text, name):
    """value of `constexpr int|long long name = <integer expression>;` (or of `#define name <integer>`), names in the
    expression resolved in `text`"""
    m = re.search(rf"constexpr\s+(?:int|long long)\s+{name}\s*=\s*([^;]+);", text)
    if m is None:
        return _define(text, name)
    expr = re.sub(r"\b([A-Za-z_]\w*)\b", lambda k: str(_const(text, k.group(1))), m.group(1).split("//")[0])
    assert re.fullmatch(r"[\d\s*+<()-]+", expr), expr
    return int(eval(expr))


def _define(text, name):
    m = re.search(rf"#define {name} (\d+)\b", text)
    assert m, name
    return int(m.group(1))


def functor_unroll(name, text=None):
    """UNROLL of `struct name` in spx_ops.cuh (a macro default resolved)"""
    text = text or _source("spx_ops.cuh")
    m = re.search(rf"struct {name} \{{.*?static constexpr int [^;]*\bUNROLL = (\w+)", text, re.S)
    assert m, name
    v = m.group(1)
    return int(v) if v.isdigit() else _define(text, v)


# the functors of the step kernels (spx_step.cu step_sep / step_box / istep_sep / istep_box)
STEP_FUNCTORS = ["ProxL1", "ProxL0", "ProxLhalf", "ProxL1Box", "ProxL0Box", "ProxLhalfBox",
                 "IproxL1", "IproxL0", "IproxL1Box", "IproxL0Box"]


def step_constants():
    ew = _source("spx_elementwise.cuh")
    return {"threads": _const(ew, "kEwThreads"), "max_partials": _const(_source("spx_common.cuh"), "kMaxPartials"),
            "unroll": {f: functor_unroll(f) for f in STEP_FUNCTORS}}


def step_grid_cap(sm_count):
    """the most CTAs step_launch gives step_kernel: 256-thread CTAs, at most 2048 threads per SM, kMaxPartials"""
    c = step_constants()
    return min(c["max_partials"], THREADS_PER_SM // c["threads"] * sm_count)


def step_tiles(n, vec, unroll):
    """tiles of step_kernel<vec, unroll> over n elements"""
    tile = step_constants()["threads"] * unroll
    return -(-(n // vec) // tile)


def step_scale_n(dt, sm_count):
    """2^k + 3: the smallest power of two at which every block of the widest tile (UNROLL = the largest of the step
    functors) runs >= 3 tiles, plus a scalar tail"""
    vec = 16 // np.dtype(dt).itemsize
    u = max(step_constants()["unroll"].values())
    k = 1
    while step_tiles(1 << k, vec, u) < 3 * step_grid_cap(sm_count):
        k += 1
    return (1 << k) + 3


def topr_routes():
    """[(largest problem length, CTA threads, keys in shared memory)] of topr_stream_launch, in order of length"""
    t = _source("spx_topr.cu")
    cap = _const(t, "kTrMaxCluster") * _const(t, "kTrChunk")
    g = re.search(r"if \(!smem_keys\) st = go\(topr_stream_kernel<R, BINF, (\d+), \d+, false, STEP>", t)
    smem = int(re.search(r"smem_keys = key_bytes <= (\d+) \* 1024;", t).group(1))
    above = re.findall(r"else if \(key_bytes > (\d+) \* 1024\) st = go\(topr_stream_kernel<R, BINF, (\d+), \d+, true, "
                       r"STEP>", t)
    last = re.search(r"else st = go\(topr_stream_kernel<R, BINF, (\d+), \d+, true, STEP>", t)
    assert "key_bytes = (size_t)n * sizeof(unsigned short)" in t  # 2 bytes of key per element
    kb = [int(a) * 1024 // 2 for a, _ in above]  # descending
    routes = [(kb[-1], int(last.group(1)), True)]
    for i in range(len(above) - 1, 0, -1):
        routes.append((kb[i - 1], int(above[i][1]), True))
    routes.append((smem * 1024 // 2, int(above[0][1]), True))
    routes.append((cap, int(g.group(1)), False))
    return routes


def topr_route(pn):
    return next((threads, smem) for top, threads, smem in topr_routes() if pn <= top)


def topr_nprob(pn, sm_count):
    """problems for >= 3 turns of every CTA's problem loop: the grid is at most sm_count x 2048 / THREADS"""
    return 3 * sm_count * (THREADS_PER_SM // topr_route(pn)[0])


def fixup_entries_per_thread():
    """what topr_step_fixup_kernel's packed count holds at most: the longest stream problem over its threads"""
    t = _source("spx_topr.cu")
    return _const(t, "kTrMaxCluster") * _const(t, "kTrChunk") // _const(t, "kFixThreads")


def binf_rounds(m, ngroups):
    """warp rounds of the uniform GroupNormL2Binf kernels: 32 / (m / kEPL) groups per round"""
    gpw = 32 // (m // _const(_source("spx_group.cu"), "kEPL"))
    return -(-ngroups // gpw), gpw


def binf_ngroups(m):
    return (1 << 23) // m + 3


def group_tasks(ngroups):
    return -(-ngroups // _const(_source("spx_group.cu"), "kTask"))


def resident_warps(sm_count):
    return THREADS_PER_SM // 32 * sm_count


TOPR_PN = [4096, 24_576, 65_536, 131_072]  # one problem length per topr_stream_kernel instance


def test_step_scale_constants_match_the_sources():
    """CPU: the thresholds, tile lengths and bounds this file derives its sizes from are the ones it was written for."""
    c = step_constants()
    assert c["threads"] == 256 and c["max_partials"] == 4736
    assert c["unroll"] == {"ProxL1": 2, "ProxL0": 2, "ProxLhalf": 2, "ProxL1Box": 2, "ProxL0Box": 2,
                           "ProxLhalfBox": 1, "IproxL1": 2, "IproxL0": 2, "IproxL1Box": 1, "IproxL0Box": 1}
    assert step_grid_cap(148) == 1184
    assert step_scale_n(np.float64, 148) == (1 << 22) + 3 and step_scale_n(np.float32, 148) == (1 << 23) + 3
    assert topr_routes() == [(18_432, 256, True), (36_864, 512, True), (102_400, 1024, True), (131_072, 512, False)]
    assert [topr_route(pn) for pn in TOPR_PN] == [(256, True), (512, True), (1024, True), (512, False)]
    assert [topr_nprob(pn, 148) for pn in TOPR_PN] == [3552, 1776, 888, 1776]
    assert fixup_entries_per_thread() == 512
    g = _source("spx_group.cu")
    assert _const(g, "kEPL") == 8 and _const(g, "kGroupThreads") == 256 and _const(g, "kTask") == 32
    for m in (16, 32, 64, 128, 256):
        nr, gpw = binf_rounds(m, binf_ngroups(m))
        assert nr >= 3 * resident_warps(148)
        assert gpw == 1 or binf_ngroups(m) % gpw != 0
    assert group_tasks(10_000_000) >= 3 * resident_warps(148)


# ---------------------------------------------------------------------------- helpers ---
def sm_count():
    p = torch.cuda.get_device_properties(0)
    assert getattr(p, "max_threads_per_multi_processor", THREADS_PER_SM) <= THREADS_PER_SM
    return p.multi_processor_count


def tdt(dt):
    return torch.float64 if dt == np.float64 else torch.float32


def dev_same(a, b):
    """bit for bit, any NaN equal to any NaN"""
    it = torch.int64 if a.dtype == torch.float64 else torch.int32
    return bool(((a.view(it) == b.view(it)) | (a.isnan() & b.isnan())).all())


def host_same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    it = np.uint64 if a.dtype == np.float64 else np.uint32
    return a.shape == b.shape and bool(np.all((a.view(it) == b.view(it)) | (np.isnan(a) & np.isnan(b))))


def scalar(x):
    return float(x.item())


def dev_sums(s, g, d=None):
    """Float64 sums of the GPU's own s on the device: Σs², Σ∇f s, Σ|∇f s| [, Σ d s², Σ|d s²|]"""
    s64, g64 = s.double(), g.double()
    gs = g64 * s64
    out = [scalar((s64 * s64).sum()), scalar(gs.sum()), scalar(gs.abs().sum())]
    if d is not None:
        ds = d.double() * s64 * s64
        out += [scalar(ds.sum()), scalar(ds.abs().sum())]
    return out


def _close(got, ref, rel, mag=None):
    if not math.isfinite(ref):
        assert (math.isnan(got) and math.isnan(ref)) or got == ref, (got, ref)
    elif mag is None:
        assert got == pytest.approx(ref, rel=rel, abs=1e-300), (got, ref)
    else:
        assert abs(got - ref) <= rel * mag, (got, ref, mag)


def check_sums(res, sums):
    """Σs² to 1e-12 relative, Σ∇f·s to 1e-12 Σ|∇f s| [, Σd s² to 1e-12 Σ|d s²|]"""
    _close(res.snorm * res.snorm if math.isfinite(res.snorm) else res.snorm, sums[0], 1e-12)
    _close(res.gdots, sums[1], 1e-12, sums[2] + 1e-300)
    if len(sums) > 3:
        _close(res.sds, sums[3], 1e-12, sums[4] + 1e-300)


def same_scalars(a, b):
    return np.asarray(tuple(a), np.float64).tobytes() == np.asarray(tuple(b), np.float64).tobytes()


def kernel_instances(fn, kernel, windows=3):
    """template argument lists of `kernel` among the CUDA kernels that `fn` launches, and every name recorded.  A
    profiling window can drop its first activities, more so right after another window closed: the calls run twice
    behind a warm-up kernel, and in a fresh window again while `kernel` is missing from the record."""
    from torch.profiler import ProfilerActivity, profile
    names = []
    for _ in range(windows):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            torch.ones(1, device=DEV).add_(1)
            torch.cuda.synchronize()
            for _ in range(2):
                fn()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        got = instances(names, kernel)
        if got:
            return got, names
    return set(), names


def instances(names, kernel):
    """template argument lists of `kernel` in demangled kernel names"""
    out = set()
    for k in names:
        m = re.search(rf"{kernel}<([^()]*)>", k)
        if m:
            out.add(tuple(a.strip().replace("(bool)1", "true").replace("(bool)0", "false") for a in m.group(1).split(",")))
    return out


def launches(fn):
    l0 = sp.launch_count()
    r = fn()
    return r, sp.launch_count() - l0


def mnu_times(g, nu):
    """fl(-ν ∇f) in the element type of ∇f, as the caller's broadcast rounds it"""
    dt = np.float64 if g.dtype == torch.float64 else np.float32
    return g * torch.tensor(dt(-dt(nu)), device=g.device)


# ===================================================================== A. step_kernel ===
H = {"l1": sp.NormL1, "l0": sp.NormL0, "lhalf": sp.RootNormLhalf}
FUNCTOR = {("step", "l1", False): "ProxL1", ("step", "l0", False): "ProxL0", ("step", "lhalf", False): "ProxLhalf",
           ("step", "l1", True): "ProxL1Box", ("step", "l0", True): "ProxL0Box", ("step", "lhalf", True): "ProxLhalfBox",
           ("istep", "l1", False): "IproxL1", ("istep", "l0", False): "IproxL0",
           ("istep", "l1", True): "IproxL1Box", ("istep", "l0", True): "IproxL0Box"}

A_CASES = ([("step", op, "sep", v, 0.0) for op in ("l1", "l0", "lhalf") for v in ("once", "twice")]
           + [("step", op, "box", v, 0.0) for op in ("l1", "l0", "lhalf") for v in ("vector", "scalar")]
           + [("istep", op, "sep", "twice", 0.25) for op in ("l1", "l0")]
           + [("istep", op, "box", "vector", ds) for op in ("l1", "l0") for ds in (0.0, 0.25)]
           + [("step", "l1", "sep", "unaligned", 0.0), ("istep", "l0", "box", "unaligned", 0.25)])


@gpu
@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("form,op,kind,variant,dshift", A_CASES, ids=["-".join(map(str, c)) for c in A_CASES])
def test_step_kernel_many_tiles(dt, form, op, kind, variant, dshift):
    """step_kernel with every block on >= 3 tiles and the last block on the scalar tail; unaligned views run
    step_kernel<1, ...> (nvec = n)."""
    sms = sm_count()
    n = step_scale_n(dt, sms)
    box, istep, unaligned = kind == "box", form == "istep", variant == "unaligned"
    functor = FUNCTOR[(form, op, box)]
    unroll = step_constants()["unroll"][functor]
    vec = 1 if unaligned else 16 // np.dtype(dt).itemsize
    cap = step_grid_cap(sms)
    assert step_tiles(n, vec, unroll) >= 3 * cap and (vec == 1 or n % vec != 0)
    lam, nu = (0.8, 0.35) if kind == "sep" else (1.0, 0.1)
    xk, sj, grad = inputs(n, dt)
    if variant == "once":
        sj = np.zeros(n, dt)
    l = u = None
    sel = osel = None
    if box:
        if variant == "scalar":
            l, u = -0.7, 0.9
        else:
            l, u = bounds(n, dt)
        if variant == "vector" and form == "step":
            sel, osel = range(1, n, 3), np.arange(1, n, 3)
    D = None
    if istep:
        D = diag(n, dt) if box else orc.uniform(n, 5, dt, 1.0, 0.5)
    # device operands: views one element into their allocations when unaligned
    put = (lambda a: T(np.concatenate([[0], a]).astype(dt))[1:]) if unaligned else T  # noqa: E731
    txk, tsj, tg = put(xk), put(sj), put(grad)
    tl = put(l) if isinstance(l, np.ndarray) else l
    tu = put(u) if isinstance(u, np.ndarray) else u
    psi = sp.shifted(H[op](lam), txk, tl, tu, selected=sel) if box else sp.shifted(H[op](lam), txk)
    if variant != "once":
        psi = sp.shifted(psi, tsj)
    new = (lambda: torch.empty(n + 1, dtype=tdt(dt), device=DEV)[1:]) if unaligned else (  # noqa: E731
        lambda: torch.empty(n, dtype=tdt(dt), device=DEV))
    s, xsy = new(), new()
    tD = put(D) if istep else None
    call = (lambda: sp.istep_(s, psi, tg, tD, dshift, xsy=xsy)) if istep else (lambda: sp.step_(s, psi, tg, nu, xsy=xsy))
    (_, res), nl = launches(call)
    assert nl == 2  # step_kernel + the fold of its partial slots
    got, names = kernel_instances(call, "step_kernel")
    assert any(a[0] == str(vec) and a[1] == str(unroll) and re.search(rf"\b{functor}<", a[2]) for a in got), names
    # the stand-alone prox!/iprox! of the same library, whole vector, on the device
    y = new()
    if istep:
        td = tD + torch.tensor(dt(dshift), device=DEV)  # d = D .+ σ rounded to R
        sp.iprox_(y, psi, tg, td)
    else:
        sp.prox_(y, psi, mnu_times(tg, nu), nu)
    assert dev_same(s, y)
    assert dev_same(xsy, (txk + tsj) + s)
    # the oracle
    gs = N(s)
    q = (dt(-dt(nu)) * grad).astype(dt)
    if istep:
        rs = solver_istep(op, xk, sj, grad, D, dshift, lam, *((l, u) if box else ()))[0]
        assert host_same(gs, rs)
    elif op != "lhalf":
        assert host_same(gs, orc.solver_step(op, xk, sj, grad, lam, nu, l, u, osel)[0])
    elif box:
        check_lhalfbox(gs, xk, sj, q, l, u, lam, nu, selected=osel, label=f"step {n}")
    else:
        ref = orc.prox_lhalf(xk, sj, q, lam, nu)
        zero = np.zeros(n, dt) - (xk + sj)
        assert np.array_equal(ref == zero, gs == zero)
        tol = 4 * np.finfo(dt).eps * (np.abs(xk) + np.abs(sj) + np.abs(q) + 1.0)
        assert np.all(np.abs(gs.astype(np.float64) - ref.astype(np.float64)) <= tol)
    # ψ(s): the L0 count exactly, the rest against the oracle's value at the GPU's s
    ref_psi = orc.value_box(op, xk, sj, gs, l, u, lam, osel) if box else orc.value_plain(op, xk, sj, gs, lam)
    _close(res.psi, ref_psi, 1e-12 if dt == np.float64 else 1e-5)
    if op == "l0":
        nz = (xsy != 0)
        if osel is not None:
            mask = torch.zeros(n, dtype=torch.bool, device=DEV)
            mask[1::3] = True
            nz &= mask
        assert res.psi == float(dt(lam) * dt(int(nz.sum().item())))
    check_sums(res, dev_sums(s, tg, (tD + torch.tensor(dt(dshift), device=DEV)) if istep else None))
    # three identical calls: the same scalars, bit for bit
    for _ in range(2):
        _, again = call()
        assert same_scalars(again, res)


# ==================================================================== B. top-r step ===
NU_T, DELTA_T = 0.3, 0.5
PLANTS = ["ties", "const", "zero", "nan", "inf"]


def plant_kind(p, nprob, pn):
    """the hard problem planted at p (every 37th and the last; at the longest length every 4th planted one is `far`:
    every element non-zero and outside the BInf ball, a flagged problem that fills the fixup kernel's packed count)"""
    if p == nprob - 1:
        return "ties"
    if p % 37:
        return None
    k = p // 37
    if pn == TOPR_PN[-1] and k % 4 == 1:
        return "far"
    return PLANTS[k % len(PLANTS)]


def plant(kind, xk, sj, g):
    """apply a planted kind to one problem's rows (numpy arrays or torch tensors, modified in place)"""
    if kind == "ties":
        xk[:] = 0; sj[:] = 0
        g[:] = (g * 2).round() / 2 if isinstance(g, torch.Tensor) else np.round(g * 2) / 2
    elif kind == "const":
        xk[:] = 0; sj[:] = 0; g[:] = 1.25
    elif kind == "zero":
        xk[:] = 0; sj[:] = 0; g[:] = 0
    elif kind == "nan":
        g[5] = float("nan"); g[-2] = float("nan")
    elif kind == "inf":
        g[9] = float("inf"); g[77] = -float("inf")
    elif kind == "far":  # z = xs + q constant (flagged); s and sj + s non-zero and |sj + s| > 1.1Δ everywhere
        xk[:] = 1.0; sj[:] = 2.0; g[:] = 1.25


def topr_host_problem(p, pn, dt, kind):
    i0 = p * pn
    xk = orc.uniform(pn, 0, dt, 4.0, -2.0, i0=i0)
    sj = orc.uniform(pn, 1, dt, 1.0, -0.5, i0=i0)
    g = orc.uniform(pn, 2, dt, 4.0, -2.0, i0=i0)
    if kind in ("psi0", "psi0_last"):  # the ψ = 0 batch: all zero but the last problem's ∇f
        xk[:] = 0; sj[:] = 0
        if kind == "psi0":
            g[:] = 0
    elif kind is not None:
        plant(kind, xk, sj, g)
    return xk, sj, g


def topr_properties(s, xk, sj, q, nprob, pn, r):
    """per problem, on the device: the kept count is min(r, #non-zero z), every kept |z| >= every dropped |z|
    (entries whose kept and dropped forms round to the same value are left out of both)"""
    xs = (xk + sj).view(nprob, pn)
    z = xs + q.view(nprob, pn)
    s = s.view(nprob, pn)
    amb = ((z - xs) == -xs) & (z != 0)
    kept = (s != -xs) & ~amb
    dropped = ~kept & ~amb
    za = torch.where(z.isnan(), torch.full_like(z, float("inf")), z.abs())
    want = (z != 0).sum(1).clamp(max=r)
    cnt = kept.sum(1)
    assert bool((cnt <= want).all()) and bool((cnt + amb.sum(1) >= want).all()), \
        torch.nonzero((cnt > want) | (cnt + amb.sum(1) < want))[:8].flatten().tolist()
    big = torch.where(kept, za, torch.full_like(za, float("inf"))).amin(1)
    small = torch.where(dropped, za, torch.zeros_like(za)).amax(1)
    assert bool((big >= small).all()), torch.nonzero(big < small)[:8].flatten().tolist()


def topr_psi_ref(s, xk, sj, xsy, r, binf, dt):
    """ψ(s) of the batch from device counts: the plain type Inf when more than r entries of xsy are non-zero, BInf also
    when an entry of sj + s lies outside the ball of 1.1Δ"""
    if not binf:
        return 0.0 if int((xsy != 0).sum().item()) <= r else math.inf
    w = sj + s
    viol = bool((w.double().abs() > 1.1 * float(dt(DELTA_T))).any())
    return math.inf if viol or int(((w + xk) != 0).sum().item()) > r else 0.0


def topr_case(dt, pn, nprob, r, xk, sj, g, kinds, grid_bound, binf, s_plain=None, check_route=False):
    """one step of the batch (plain or BInf) through every bar; returns s"""
    psi = sp.shifted(sp.IndBallL0(r), xk, DELTA_T, sp.NormLinf(1.0), nprob=nprob) if binf else \
        sp.shifted(sp.IndBallL0(r), xk, nprob=nprob)
    psi = sp.shifted(psi, sj)
    s, xsy = torch.empty_like(g), torch.empty_like(g)
    call = lambda: sp.step_(s, psi, g, NU_T, xsy=xsy)  # noqa: E731
    (_, res), nl = launches(call)
    assert nl == 4  # stream step kernel, radix kernel on the flagged problems, fixup kernel, fold
    if check_route:
        threads, smem = topr_route(pn)
        want = ("double" if dt == np.float64 else "float", "true" if binf else "false", str(threads), None,
                "true" if smem else "false", "true")
        got, _ = kernel_instances(call, "topr_stream_kernel")
        assert any(all(w is None or w == a for w, a in zip(want, inst)) for inst in got), (want, got)
    q = mnu_times(g, NU_T)
    y = torch.empty_like(g)
    sp.prox_(y, psi, q, NU_T)
    assert dev_same(s, y)
    assert dev_same(xsy, (xk + sj) + s)
    if binf:
        assert dev_same(s, s_plain.clamp(-DELTA_T, DELTA_T))
    else:
        topr_properties(s, xk, sj, q, nprob, pn, r)
    ref_psi = topr_psi_ref(s, xk, sj, xsy, r, binf, dt)
    assert res.psi == ref_psi and res.psi == psi(s)
    check_sums(res, dev_sums(s, g))
    for _ in range(2):
        _, again = sp.step_(s, psi, g, NU_T, xsy=xsy)
        assert same_scalars(again, res)
    # whole problems against the oracle: first, last, every planted kind, two past the grid
    probe = {0, nprob - 1}
    for k in set(kinds.values()):
        probe.add(min(p for p, v in kinds.items() if v == k))
    past = [p for p in range(grid_bound + 1, nprob) if p not in kinds]
    probe.update(past[:1] + past[-1:])
    for p in sorted(probe):
        hxk, hsj, hg = topr_host_problem(p, pn, dt, kinds.get(p))
        hq = (dt(-dt(NU_T)) * hg).astype(dt)
        ref = orc.prox_indballl0(hxk, hsj, hq, r, delta=DELTA_T if binf else None)
        assert host_same(N(s[p * pn:(p + 1) * pn]), ref), (p, kinds.get(p))
    return s


def topr_batch(dt, nprob, pn, kinds):
    """device inputs of the batch (the hash generator, streams 0-2), hard problems planted"""
    n = nprob * pn
    f = tdt(dt)
    xk, sj, g = dev_uniform(n, 0, f, 4.0, -2.0), dev_uniform(n, 1, f, 1.0, -0.5), dev_uniform(n, 2, f, 4.0, -2.0)
    xv, sv, gv = xk.view(nprob, pn), sj.view(nprob, pn), g.view(nprob, pn)
    for p, kind in kinds.items():
        plant(kind, xv[p], sv[p], gv[p])
    return xk, sj, g


@gpu
@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("pn", TOPR_PN)
def test_step_topr_every_instance_with_the_problem_loop(dt, pn):
    """The top-r step on each topr_stream_kernel instance, every CTA walking >= 3 problems: an ordinary batch (r = 1024;
    also r = 1 and r = pn - 1 on the global-key instance), hard problems every 37th and last (radix + fixup kernels),
    and a batch whose only non-zero problem is the last (ψ = 0).  Plain and BInf."""
    sms = sm_count()
    threads, _ = topr_route(pn)
    nprob = topr_nprob(pn, sms)
    grid_bound = sms * (THREADS_PER_SM // threads)
    assert nprob >= 3 * grid_bound
    if pn == TOPR_PN[-1]:
        assert pn // 256 == fixup_entries_per_thread()  # the `far` problem fills the fixup kernel's count
    rs = [1024] + ([1, pn - 1] if pn == TOPR_PN[-1] else [])
    # ordinary batches
    xk, sj, g = topr_batch(dt, nprob, pn, {})
    for r in rs:
        sp_ = topr_case(dt, pn, nprob, r, xk, sj, g, {}, grid_bound, False, check_route=(r == rs[0]))
        topr_case(dt, pn, nprob, r, xk, sj, g, {}, grid_bound, True, s_plain=sp_, check_route=(r == rs[0]))
        del sp_
    # hard problems spread over the grid
    kinds = {p: k for p in range(nprob) if (k := plant_kind(p, nprob, pn)) is not None}
    assert set(kinds.values()) >= set(PLANTS) and any(p >= grid_bound for p in kinds)
    del xk, sj, g
    xk, sj, g = topr_batch(dt, nprob, pn, kinds)
    sp_ = topr_case(dt, pn, nprob, 1024, xk, sj, g, kinds, grid_bound, False)
    topr_case(dt, pn, nprob, 1024, xk, sj, g, kinds, grid_bound, True, s_plain=sp_)
    del sp_, xk, sj, g
    # ψ = 0: zeros except the last problem's ∇f (reached on a later turn of the loop)
    f = tdt(dt)
    n = nprob * pn
    xk, sj = torch.zeros(n, dtype=f, device=DEV), torch.zeros(n, dtype=f, device=DEV)
    g = torch.zeros(n, dtype=f, device=DEV)
    g[(nprob - 1) * pn:] = dev_uniform(pn, 2, f, 4.0, -2.0, i0=(nprob - 1) * pn)
    kinds = {p: "psi0" for p in range(nprob - 1)}
    kinds[nprob - 1] = "psi0_last"
    sp_ = topr_case(dt, pn, nprob, 1024, xk, sj, g, kinds, grid_bound, False)
    topr_case(dt, pn, nprob, 1024, xk, sj, g, kinds, grid_bound, True, s_plain=sp_)


# =========================================================== C. the group steps ===
NU_G, DELTA_G = 0.3, 0.5


def group_windows(ng, wg, rng, extra=()):
    return sorted({0, ng - wg, *(int(o) for o in rng.integers(0, ng - wg, size=3)), *extra})


def binf_psi64(s, xk, sj, lam_g, m, dt):
    """ψ(s) of GroupNormL2Binf on a uniform layout from the GPU's s, in the step kernel's association -- v = (sj + s) + xk
    in R, λ_g ‖v_g‖ rounded to R, the terms summed in Float64 -- and Inf outside the ball of 1.1Δ"""
    w = sj + s
    if bool((w.double().abs() > 1.1 * float(dt(DELTA_G))).any()):
        return math.inf
    v = (w + xk).double().view(-1, m)
    terms = lam_g * torch.sqrt((v * v).sum(1)).to(s.dtype)
    return float(dt(scalar(terms.double().sum())))


@gpu
@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("m", [16, 32, 64, 128, 256])
def test_step_groupl2binf_uniform_many_rounds(dt, m):
    """The one-pass GroupNormL2Binf step with every warp on >= 3 rounds (the FAST form's double buffer flips at least
    twice) and a partial last round; `huge` and `big_lambda` send rounds across the whole range to the list form."""
    sms = sm_count()
    ng = binf_ngroups(m)
    n = ng * m
    nrounds, gpw = binf_rounds(m, ng)
    assert nrounds >= 3 * resident_warps(sms) and (gpw == 1 or ng % gpw != 0)
    xk, sj, grad = inputs(n, dt)
    lam0 = (dt(0.5) + orc.uniform(ng, 12, dt)).astype(dt)
    offs = np.arange(0, n + 1, m)
    txk, tsj, toffs = T(xk), T(sj), T(offs)
    rng = np.random.default_rng(m)
    wg = 2000
    for regime in ("base", "huge", "big_lambda"):
        g, lam_g = grad, lam0
        if regime == "huge":  # |sol| ~ 1e13 on every 97th group: beyond the Float32 guards of the fast search
            g = grad.copy()
            for gi in range(5, ng, 97):
                g[gi * m:(gi + 1) * m] *= dt(1e13)
        elif regime == "big_lambda":
            lam_g = (lam0 * dt(200.0)).astype(dt)
        tg = T(g)
        psi = sp.shifted(sp.shifted(sp.GroupNormL2(T(lam_g), None, offsets=toffs), txk, DELTA_G, sp.NormLinf(1.0)), tsj)
        s, xsy = torch.empty_like(tg), torch.empty_like(tg)
        call = lambda: sp.step_(s, psi, tg, NU_G, xsy=xsy)  # noqa: E731
        (_, res), nl = launches(call)
        assert nl == 4  # layout check, FAST and list forms, fold
        if regime == "base":
            got, _ = kernel_instances(call, "group_l2binf_uniform_kernel")
            assert (("double" if dt == np.float64 else "float"), str(m // 8), "true", "true") in got, got
        y = torch.empty_like(tg)
        sp.prox_(y, psi, mnu_times(tg, NU_G), NU_G)
        assert dev_same(s, y)
        assert dev_same(xsy, (txk + tsj) + s)
        gs = N(s)
        _close(res.psi, binf_psi64(s, txk, tsj, T(lam_g), m, dt), 1e-12 if dt == np.float64 else 1e-5)
        if dt == np.float64:  # the oracle sums ψ in R: in Float32 its own rounding reaches 1e-5 at this size
            _close(res.psi, orc.value_binf("groupl2", xk, sj, gs, DELTA_G, offs=offs, lam_g=lam_g), 1e-12)
        check_sums(res, dev_sums(s, tg))
        for _ in range(2):
            _, again = call()
            assert same_scalars(again, res)
        q = (dt(-dt(NU_G)) * g).astype(dt)
        planted = 5 + 97 * (ng // 2 // 97)  # a `huge` group in the middle of the range
        for g0 in group_windows(ng, wg, rng, extra=(planted - wg // 2,)):
            # the groups of the window; in the `huge` regime without the planted groups themselves: their s is a
            # difference of ~1e12 magnitudes, which neither support nor 8 ulp of the scale can pin down (it is pinned
            # to prox! above), while their neighbours in the same declined rounds are checked here
            keep = np.array([regime != "huge" or (gi - 5) % 97 != 0 for gi in range(g0, g0 + wg)])
            el = np.repeat(keep, m)
            a, b = g0 * m, (g0 + wg) * m
            check_groupl2binf(gs[a:b][el], xk[a:b][el], sj[a:b][el], q[a:b][el], np.arange(0, int(el.sum()) + 1, m),
                              lam_g[g0:g0 + wg][keep], NU_G, DELTA_G, label=f"{regime} m={m} window {g0}")


@gpu
@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("layout", ["g64", "short_ragged"])
def test_step_groupl2_single_pass_at_scale(dt, layout):
    """The one-pass GroupNormL2 step (group_l2_step_kernel) at 2^23 elements: the bars of
    test_step_groupl2_single_pass_on_short_group_layouts, its composed form (SPX_STEP_COMPOSED) giving the same s, and
    windows of whole groups against the oracle at 8 ulp of the value scale."""
    rng = np.random.default_rng(7)
    sizes = np.full((1 << 23) // 64 + 3, 64) if layout == "g64" else rng.integers(1, 257, (1 << 23) // 128 + 3)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    ng, n = sizes.size, int(offs[-1])
    xk, sj, grad = inputs(n, dt)
    lam_g = (dt(0.5) + orc.uniform(ng, 12, dt)).astype(dt)
    txk, tsj, tg = T(xk), T(sj), T(grad)
    psi = sp.shifted(sp.shifted(sp.GroupNormL2(T(lam_g), None, offsets=T(offs)), txk), tsj)
    s, xsy = torch.empty_like(tg), torch.empty_like(tg)
    call = lambda: sp.step_(s, psi, tg, NU_G, xsy=xsy)  # noqa: E731
    (_, res), nl = launches(call)
    assert nl == 2  # group_l2_step_kernel + fold
    y = torch.empty_like(tg)
    sp.prox_(y, psi, mnu_times(tg, NU_G), NU_G)
    assert dev_same(s, y)
    assert dev_same(xsy, (txk + tsj) + s)
    gs = N(s)
    _close(res.psi, orc.value_groupl2(xk, sj, gs, offs, lam_g), 1e-12 if dt == np.float64 else 1e-5)
    check_sums(res, dev_sums(s, tg))
    for _ in range(2):
        _, again = call()
        assert same_scalars(again, res)
    s_fused = s.clone()
    os.environ["SPX_STEP_COMPOSED"] = "1"
    try:
        (_, res_c), nl = launches(call)
    finally:
        del os.environ["SPX_STEP_COMPOSED"]
    assert nl > 2 and torch.equal(s, s_fused)
    q = (dt(-dt(NU_G)) * grad).astype(dt)
    eps = np.finfo(dt).eps
    for g0 in group_windows(ng, 2000, rng):
        a, b = int(offs[g0]), int(offs[g0 + 2000])
        ref = orc.prox_groupl2(xk[a:b], sj[a:b], q[a:b], offs[g0:g0 + 2001] - a, lam_g[g0:g0 + 2000], NU_G)
        scale = np.abs(xk[a:b]).astype(np.float64) + np.abs(sj[a:b]) + np.abs(q[a:b]) + 1
        assert np.all(np.abs(gs[a:b].astype(np.float64) - ref) <= 8 * eps * scale), (layout, g0)


# ============================================================ D. the BASELINE shapes ===
CHUNK = 1 << 22


def stream_chunks(n, fn):
    """fn(i0, m) over the chunks of [0, n), in threads (the oracle and numpy release the GIL); results in order"""
    spans = [(i0, min(CHUNK, n - i0)) for i0 in range(0, n, CHUNK)]
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        return list(ex.map(lambda a: fn(*a), spans))


def fold64(vals):
    return sum(vals) % (1 << 64)


@gpu
def test_c1_step_l1_at_2p28():
    """C1's step: ShiftedNormL1 shifted once, n = 2^28 Float64: whole-vector checksums of s and xsy against the streamed
    oracle step, scalars against chunked Float64 sums."""
    n = 1 << (28 - SHRINK)
    assert step_tiles(n, 2, step_constants()["unroll"]["ProxL1"]) >= 3 * step_grid_cap(sm_count())
    lam, nu = 1.0, 0.1
    xk, g = dev_uniform(n, 0, scale=4.0, shift=-2.0), dev_uniform(n, 2, scale=4.0, shift=-2.0)
    psi = sp.shifted(sp.NormL1(lam), xk)
    s, xsy = torch.empty_like(g), torch.empty_like(g)
    _, res = sp.step_(s, psi, g, nu, xsy=xsy)
    got = (dev_checksum(s), dev_checksum(xsy))

    def chunk(i0, m):
        hxk = orc.uniform(m, 0, np.float64, 4.0, -2.0, i0=i0)
        hg = orc.uniform(m, 2, np.float64, 4.0, -2.0, i0=i0)
        rs, rxsy, rpsi, _, _ = orc.solver_step("l1", hxk, np.zeros(m), hg, lam, nu)
        gs = hg * rs
        return (host_checksum(rs, i0), host_checksum(rxsy, i0), rpsi, float(np.sum(rs * rs)), float(np.sum(gs)),
                float(np.sum(np.abs(gs))))

    parts = stream_chunks(n, chunk)
    assert got == (fold64(p[0] for p in parts), fold64(p[1] for p in parts))
    _close(res.psi, math.fsum(p[2] for p in parts), 1e-12)
    check_sums(res, [math.fsum(p[k] for p in parts) for k in (3, 4, 5)])


@gpu
def test_c2_istep_l0box_at_2p28():
    """The C2 operands through istep_ of ShiftedNormL0Box (vector bounds, the diagonal with negative and zero entries,
    dshift = 0.25), n = 2^28 Float64: checksums of s and xsy against the streamed oracle istep, ψ (a count) exactly."""
    n = 1 << (28 - SHRINK)
    assert step_tiles(n, 2, step_constants()["unroll"]["IproxL0Box"]) >= 3 * step_grid_cap(sm_count())
    lam, dshift = 1.0, 0.25
    xk, sj, g = dev_uniform(n, 0, scale=4.0, shift=-2.0), dev_uniform(n, 1, shift=-0.5), dev_uniform(n, 2, scale=4.0, shift=-2.0)
    l = dev_uniform(n, 3).add_(0.25).neg_()
    u = dev_uniform(n, 4).add_(0.25)
    D = dev_uniform(n, 5).add_(0.5)
    b = dev_uniform(n, 6)
    D = torch.where(b < 0.1, -D, D)
    D = torch.where((b >= 0.1) & (b < 0.2), torch.zeros_like(D), D)
    del b
    psi = sp.shifted(sp.shifted(sp.NormL0(lam), xk, l, u), sj)
    s, xsy = torch.empty_like(g), torch.empty_like(g)
    _, res = sp.istep_(s, psi, g, D, dshift, xsy=xsy)
    got = (dev_checksum(s), dev_checksum(xsy))

    def chunk(i0, m):
        hxk, hsj, hg, hl, hu, hD = c2_host_inputs(i0, m)
        rs, rxsy, rpsi, _, _, _ = solver_istep("l0", hxk, hsj, hg, hD, dshift, lam, hl, hu)
        d = hD + dshift
        gs, ds = hg * rs, d * rs * rs
        return (host_checksum(rs, i0), host_checksum(rxsy, i0), rpsi, float(np.sum(rs * rs)), float(np.sum(gs)),
                float(np.sum(np.abs(gs))), float(np.sum(ds)), float(np.sum(np.abs(ds))))

    parts = stream_chunks(n, chunk)
    assert got == (fold64(p[0] for p in parts), fold64(p[1] for p in parts))
    assert res.psi == math.fsum(p[2] for p in parts)  # λ = 1: the count of non-zeros, exactly
    check_sums(res, [math.fsum(p[k] for p in parts) for k in (3, 4, 5, 6, 7)])


@gpu
def test_c4_group_steps_10m_groups_of_64():
    """C4: step_ of ShiftedGroupNormL2 (one pass, every warp on >= 3 tasks) and ShiftedGroupNormL2Binf (uniform layout,
    >= 3 rounds per warp) on 10^7 groups of 64 Float64: whole-vector s == prox! and xsy on the device, scalars against
    Float64 sums, windows of whole groups against the oracle."""
    sms = sm_count()
    gs_ = 64
    ng = max(10_000_000 >> SHRINK, 3 * resident_warps(sms) * 32)
    assert group_tasks(ng) >= 3 * resident_warps(sms) and binf_rounds(gs_, ng)[0] >= 3 * resident_warps(sms)
    n = ng * gs_
    xk, sj, g = dev_uniform(n, 0, scale=4.0, shift=-2.0), dev_uniform(n, 1, shift=-0.5), dev_uniform(n, 2, scale=4.0, shift=-2.0)
    lam_g = dev_uniform(ng, 12, shift=0.5)
    offs = torch.arange(0, n + 1, gs_, dtype=torch.int64, device=DEV)
    h = sp.GroupNormL2(lam_g, None, offsets=offs)
    q = mnu_times(g, NU_G)
    rng = np.random.default_rng(9)
    eps = np.finfo(np.float64).eps
    for binf in (False, True):
        psi = sp.shifted(sp.shifted(h, xk, DELTA_G, sp.NormLinf(1.0)), sj) if binf else sp.shifted(sp.shifted(h, xk), sj)
        s, xsy = torch.empty_like(g), torch.empty_like(g)
        (_, res), nl = launches(lambda: sp.step_(s, psi, g, NU_G, xsy=xsy))
        assert nl == (4 if binf else 2)
        y = torch.empty_like(g)
        sp.prox_(y, psi, q, NU_G)
        assert dev_same(s, y)
        del y
        assert dev_same(xsy, (xk + sj) + s)
        assert res.psi == pytest.approx(psi(s), rel=1e-12)
        check_sums(res, dev_sums(s, g))
        wg = 2000
        for g0 in group_windows(ng, wg, rng):
            i0, m = g0 * gs_, wg * gs_

            def u(k, **kw):
                return orc.uniform(m, k, np.float64, i0=i0, **kw)
            hxk, hsj, hg = u(0, scale=4.0, shift=-2.0), u(1, shift=-0.5), u(2, scale=4.0, shift=-2.0)
            hq = -0.3 * hg
            hlam = orc.uniform(wg, 12, np.float64, shift=0.5, i0=g0)
            ho = np.arange(0, m + 1, gs_)
            got = N(s[i0:i0 + m])
            if binf:
                check_groupl2binf(got, hxk, hsj, hq, ho, hlam, NU_G, DELTA_G, label=f"C4 step window {g0}")
            else:
                ref = orc.prox_groupl2(hxk, hsj, hq, ho, hlam, NU_G)
                scale = np.abs(hxk) + np.abs(hsj) + np.abs(hq) + 1
                assert np.all(np.abs(got - ref) <= 8 * eps * scale), g0
        del s, xsy


@gpu
def test_c5_topr_step_4096_problems():
    """C5: step_ of ShiftedIndBallL0 and ShiftedIndBallL0BInf, 4096 problems of 65536 Float64, r = 1024, one pass of
    the stream kernel: per-problem properties on the device, three whole problems against the oracle."""
    sms = sm_count()
    pn, r = 65_536, 1024
    nprob = max(4096 >> SHRINK, topr_nprob(pn, sms))
    grid_bound = sms * (THREADS_PER_SM // topr_route(pn)[0])
    assert nprob >= 3 * grid_bound
    xk, sj, g = topr_batch(np.float64, nprob, pn, {})
    # topr_case probes the first and last problems and two past the grid
    s_plain = topr_case(np.float64, pn, nprob, r, xk, sj, g, {}, grid_bound, False, check_route=True)
    topr_case(np.float64, pn, nprob, r, xk, sj, g, {}, grid_bound, True, s_plain=s_plain, check_route=True)


@gpu
def test_step_l1_f32_past_2p31_elements():
    """step_ of ShiftedNormL1, Float32, n = 2^31 + 5: element indices past 2^31 in step_kernel.  Windows against the
    oracle at the start, across element 2^31 and at the tail; whole-vector s == prox! and xsy on the device; the sums
    against chunked Float64 sums."""
    n = (1 << (31 - SHRINK)) + 5
    f = torch.float32
    lam, nu = 1.0, 0.1
    xk, g = dev_uniform(n, 0, f, 4.0, -2.0), dev_uniform(n, 2, f, 4.0, -2.0)
    psi = sp.shifted(sp.NormL1(lam), xk)
    s, xsy = torch.empty_like(g), torch.empty_like(g)
    _, res = sp.step_(s, psi, g, nu, xsy=xsy)
    # the stand-alone prox! in place over fl(-ν ∇f): the fifth vector
    q = mnu_times(g, nu)
    sp.prox_(q, psi, q, nu)
    assert dev_same(s, q)
    del q
    w = 1 << 16
    for i0 in (0, (1 << (31 - SHRINK)) - w + 1, n - w):  # the middle window ends on element 2^31
        hxk = orc.uniform(w, 0, np.float32, 4.0, -2.0, i0=i0)
        hg = orc.uniform(w, 2, np.float32, 4.0, -2.0, i0=i0)
        rs, rxsy, _, _, _ = orc.solver_step("l1", hxk, np.zeros(w, np.float32), hg, lam, nu)
        assert host_same(N(s[i0:i0 + w]), rs) and host_same(N(xsy[i0:i0 + w]), rxsy), i0
    parts = []
    step = 1 << 27
    for a in range(0, n, step):
        xs, ss, gg, xx = s[a:a + step], xsy[a:a + step], g[a:a + step], xk[a:a + step]
        assert dev_same(ss, (xx + 0.0) + xs)
        s64, gs = xs.double(), gg.double() * xs.double()
        parts.append((scalar(ss.double().abs().sum()), scalar((s64 * s64).sum()), scalar(gs.sum()), scalar(gs.abs().sum())))
    _close(res.psi, lam * math.fsum(p[0] for p in parts), 1e-5)
    check_sums(res, [math.fsum(p[k] for p in parts) for k in (1, 2, 3)])
