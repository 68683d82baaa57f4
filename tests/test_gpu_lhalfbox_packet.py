"""ShiftedRootNormLhalfBox prox! through ew_kernel's packet path (the vector launches: every element of a 128-bit packet
filtered as straight-line code, the hard ones patched with the exact form afterwards, the next packet's loads in flight)
against the per-element path of the same operands: a one-element-offset view (the VEC = 1 launch) and the fused step's
`s` (step_kernel).  Both must give the same y bit for bit, on data where no element, one element per packet or every
element needs the exact form."""
import numpy as np
import pytest
import torch

LAM, SIGMA = 1.0, 0.1
DT = [np.float64, np.float32]


def _gpu():
    from gpu_util import DEV, N, T, bounds, check_lhalfbox, inputs, sp
    return DEV, N, T, bounds, check_lhalfbox, inputs, sp


def _hard_rows(dt, sigma):
    """(xk, sj, q, l, u) rows the Float32 filter cannot decide: exact ties, t within 0.2 % of 1, non-finite operands,
    |xk + sj + q| outside the Float32-friendly range"""
    z1 = 3.0 * (sigma * LAM / 4.0) ** (2.0 / 3.0)  # |xk + sj + q| at t = 1
    rows = [(0.0, 0.0, 0.0, -1.0, 1.0), (0.0, 0.0, 0.0, -0.5, 0.5), (0.25, -0.25, 0.0, -2.0, 2.0)]
    for f in (1.0, 1.0 + 1e-4, 1.0 - 1e-4, 1.0 + 1e-3, 1.0 - 1e-3):
        rows += [(0.1, 0.05, z1 * f - 0.15, -1.0, 1.0), (-0.1, -0.05, -z1 * f + 0.15, -1.0, 1.0)]
    nan, inf = np.nan, np.inf
    rows += [(nan, 0.1, 0.2, -1.0, 1.0), (0.1, nan, 0.2, -1.0, 1.0), (0.1, 0.2, nan, -1.0, 1.0),
             (0.1, 0.2, 0.3, nan, 1.0), (0.1, 0.2, 0.3, -1.0, nan), (inf, 0.0, 0.0, -1.0, 1.0),
             (0.0, -inf, 0.0, -1.0, 1.0), (0.0, 0.0, inf, -1.0, 1.0), (0.0, 0.0, -inf, -inf, inf),
             (0.0, 0.0, 1e-12, -1.0, 1.0), (0.0, 0.0, -3e-10, -1.0, 1.0), (1e12, 0.0, 0.5, -1e13, 1e13),
             (0.0, 2e9, -1.0, -1e10, 1e10)]
    if dt == np.float64:
        rows += [(1e300, 0.0, 1e300, -1e308, 1e308), (0.0, 0.0, 1e-300, -1.0, 1.0)]
    return np.asarray(rows, dtype=dt)


def _operands(case, n, dt):
    _, _, _, bounds, _, inputs, _ = _gpu()
    xk, sj, q = inputs(n, dt)
    l, u = bounds(n, dt)
    ops = np.stack([xk, sj, q, l, u])
    if case == "regular":
        return ops
    rows = _hard_rows(dt, SIGMA)
    vec = 16 // np.dtype(dt).itemsize
    if case == "all_hard":
        pos = np.arange(n)
    else:  # one element in every third packet, its place in the packet rotating
        p = np.arange(0, n // vec, 3)
        pos = p * vec + (p // 3) % vec
    ops[:, pos] = rows[np.arange(pos.size) % len(rows)].T
    return ops


def _bits(a):
    return a.view(np.uint64 if a.dtype == np.float64 else np.uint32)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DT)
@pytest.mark.parametrize("case", ["regular", "all_hard", "one_hard"])
@pytest.mark.parametrize("n", [4099, (1 << 21) + 3])  # a scalar tail for both packet widths; several grid-stride sweeps
@pytest.mark.parametrize("selk", [None, "range"])
def test_lhalfbox_packet_matches_per_element(dt, case, n, selk):
    DEV, N, T, _, check_lhalfbox, _, sp = _gpu()
    xk, sj, q, l, u = _operands(case, n, dt)
    sel_dev, sel_host = (None, None) if selk is None else (range(1, n, 3), np.arange(1, n, 3))
    off = lambda a: T(np.concatenate([a[:1], a]))[1:]  # noqa: E731  (one element past a 16-byte boundary)
    tq = T(q)
    psi = sp.shifted(sp.shifted(sp.RootNormLhalf(LAM), T(xk), T(l), T(u), sel_dev), T(sj))
    assert tq.data_ptr() % 16 == 0
    y = torch.empty_like(tq)
    sp.prox_(y, psi, tq, SIGMA)
    got = N(y)

    # per element: the same operands through the VEC = 1 launch
    psi_off = sp.shifted(sp.shifted(sp.RootNormLhalf(LAM), off(xk), off(l), off(u), sel_dev), off(sj))
    y_off = off(np.zeros(n, dt))
    sp.prox_(y_off, psi_off, off(q), SIGMA)
    assert np.array_equal(_bits(got), _bits(N(y_off))), np.flatnonzero(_bits(got) != _bits(N(y_off)))[:5]

    # the fused-ψ form: the same y
    y_psi = torch.empty_like(tq)
    _, v = sp.prox_(y_psi, psi, tq, SIGMA, want_value=True)
    assert np.array_equal(_bits(got), _bits(N(y_psi)))
    _, v_off = sp.prox_(y_off, psi_off, off(q), SIGMA, want_value=True)
    if np.isnan(v) or np.isnan(v_off) or np.isinf(v) or np.isinf(v_off):
        assert np.asarray(v).tobytes() == np.asarray(v_off).tobytes() or (np.isnan(v) and np.isnan(v_off)), (v, v_off)
    else:  # one partial per CTA: the two launches sum in different orders
        assert abs(v - v_off) <= (1e-12 if dt == np.float64 else 2e-6) * max(1.0, abs(v_off)), (v, v_off)

    # in place, y is q
    yq = tq.clone()
    sp.prox_(yq, psi, yq, SIGMA)
    assert np.array_equal(_bits(got), _bits(N(yq)))

    # the fused step (step_kernel, per element): s = prox!(-ν ∇f, ν) with ∇f = -q and ν = σ = 1 (exact negation)
    y1 = torch.empty_like(tq)
    sp.prox_(y1, psi, tq, 1.0)
    s = torch.empty_like(tq)
    sp.step_(s, psi, -tq, 1.0)
    assert np.array_equal(_bits(N(y1)), _bits(N(s))), np.flatnonzero(_bits(N(y1)) != _bits(N(s)))[:5]

    if case == "regular":
        check_lhalfbox(got, xk, sj, q, l, u, LAM, SIGMA, selected=sel_host, label=f"packet {dt.__name__} n={n}")
