#!/usr/bin/env python
"""Per-operator device-resident timing of every in-scope prox!/iprox!/ψ(y) (SURVEY.md §8d configs).

    python tools/bench_ops.py [--log2n 28] [--dtype f64] [--reps 10] [--only REGEX] [--json out.json]

Prints one line per operator: ms, elements/s, algorithmic GB/s, fraction of the measured HBM peak.
CUDA events on the launching stream, 3 warm-ups, operands far larger than L2.
"""
import argparse
import json
import os
import re
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "shiftedproximaloperators.jl_b200"))
import ctypes as C  # noqa: E402

import shiftedprox as sp  # noqa: E402
from shiftedprox import _lib as L  # noqa: E402

SEED = 20261018


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", type=int, default=28)
    ap.add_argument("--dtype", default="f64")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--only", default=".*")
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    tdt = torch.float64 if args.dtype == "f64" else torch.float32
    R = 8 if args.dtype == "f64" else 4
    n = 1 << args.log2n
    try:
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        peak = 6650.0

    def uni(stream, scale=1.0, shift=0.0, m=n):
        t = torch.empty(m, dtype=tdt, device=dev)
        f = f"spx_fill_uniform_{args.dtype}"
        ct = C.c_double if args.dtype == "f64" else C.c_float
        L.call(f, sp.context(dev), C.c_void_p(t.data_ptr()), C.c_int64(m), C.c_int64(0), C.c_uint64(SEED),
               C.c_uint64(stream), ct(scale), ct(shift))
        return t

    xk, sj, q = uni(0, 4.0, -2.0), uni(1, 1.0, -0.5), uni(2, 4.0, -2.0)
    l = uni(3).add_(0.25).neg_()
    u = uni(4).add_(0.25)
    d = uni(5).add_(0.5)
    b = uni(6)
    dpos = d.clone()
    d = torch.where(b < 0.1, -d, d)
    d = torch.where((b >= 0.1) & (b < 0.2), torch.zeros_like(d), d)
    del b
    y = torch.empty(n, dtype=tdt, device=dev)
    lam, sigma = 1.0, 0.1
    results = []

    def timeit(name, fn, alg_bytes_per_elt, elems=n, note=""):
        if not re.search(args.only, name):
            return
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.reps)]
        for a, b_ in ev:
            a.record()
            fn()
            b_.record()
        torch.cuda.synchronize()
        ts = sorted(a.elapsed_time(b_) for a, b_ in ev)
        ms = ts[len(ts) // 2]
        gbs = alg_bytes_per_elt * elems / (ms * 1e-3) / 1e9
        r = {"op": name, "dtype": args.dtype, "n": elems, "ms_median": ms, "ms_best": ts[0],
             "elements_per_s": elems / (ms * 1e-3), "alg_bytes_per_elt": alg_bytes_per_elt, "GBps": gbs,
             "frac_measured_peak": gbs / peak, "frac_nominal_8000": gbs / 8000.0, "note": note}
        results.append(r)
        print(f"{name:34s} {ms:9.3f} ms  {r['elements_per_s']:.3e} el/s  {gbs:8.1f} GB/s  "
              f"{100 * gbs / peak:5.1f}% of measured {peak:.0f}  {note}", flush=True)

    def step_pair(name, psi, composed_transits, note):
        # spx_step_groupl2 (5 vector transits; 8 on one group) against ShiftedProximableFunction.step_ of the same ψ:
        # first whether both give the same s and xsy bit for bit, then both timed, alternated three times (q plays ∇f)
        xsy_a, s_b, xsy_b = torch.empty_like(y), torch.empty_like(y), torch.empty_like(y)
        _, r = sp.step_(y, psi, q, 0.3, xsy=xsy_a)
        _, r2 = sp.ShiftedProximableFunction.step_(psi, s_b, q, 0.3, xsy=xsy_b)
        same = torch.equal(y, s_b) and torch.equal(xsy_a, xsy_b)
        print(f"{name} vs composed: s and xsy bit-identical: {same}; scalars {tuple(r)} vs {tuple(r2)}", flush=True)
        del s_b, xsy_b
        fused = 8 if name.endswith("_one") else 5
        for _ in range(3):
            timeit(name, lambda: sp.step_(y, psi, q, 0.3, xsy=xsy_a), fused * R,
                   note=f"spx_step_groupl2, {note}; alg. bytes = {fused} transits")
            timeit(f"{name}_composed", lambda: sp.ShiftedProximableFunction.step_(psi, y, q, 0.3, xsy=xsy_a),
                   fused * R, note=f"step_pre, prox! in place + ψ, step_post ({composed_transits} transits); "
                                  "alg. bytes as above")
        del xsy_a

    def two(h, *a, **k):
        return sp.shifted(sp.shifted(h, xk, *a, **k), sj)

    # separable
    for nm, h in (("l1", sp.NormL1(lam)), ("l0", sp.NormL0(lam)), ("lhalf", sp.RootNormLhalf(lam))):
        psi = two(h)
        timeit(f"prox_{nm}", lambda psi=psi: sp.prox_(y, psi, q, sigma), 4 * R)
        timeit(f"prox_{nm}+psi", lambda psi=psi: sp.prox_(y, psi, q, sigma, want_value=True), 4 * R, note="fused ψ(y)")
        timeit(f"value_{nm}", lambda psi=psi: psi(y), 3 * R)
        if nm != "lhalf":
            timeit(f"iprox_{nm}", lambda psi=psi: sp.iprox_(y, psi, q, dpos), 5 * R)
    # Box, vector bounds and scalar bounds
    for nm, h in (("l1box", sp.NormL1(lam)), ("l0box", sp.NormL0(lam)), ("lhalfbox", sp.RootNormLhalf(lam))):
        psi = two(h, l, u)
        timeit(f"prox_{nm}_vec", lambda psi=psi: sp.prox_(y, psi, q, sigma), 6 * R)
        timeit(f"prox_{nm}_vec+psi", lambda psi=psi: sp.prox_(y, psi, q, sigma, want_value=True), 6 * R, note="fused ψ(y)")
        psis = two(h, -1.0, 1.0)
        timeit(f"prox_{nm}_scalar", lambda psi=psis: sp.prox_(y, psi, q, sigma), 4 * R)
        psir = two(h, l, u, range(0, n, 2))
        timeit(f"prox_{nm}_vec_sel1:2:n", lambda psi=psir: sp.prox_(y, psi, q, sigma), 6 * R)
        timeit(f"value_{nm}_vec", lambda psi=psi: psi(y), 5 * R)
        if nm != "lhalfbox":
            timeit(f"iprox_{nm}_vec", lambda psi=psi: sp.iprox_(y, psi, q, d), 7 * R)
            timeit(f"iprox_{nm}_scalar", lambda psi=psis: sp.iprox_(y, psi, q, d), 5 * R)
    # fused solver step (SURVEY.md §8f rank 1): q = -ν∇f, prox!, ψ(s), xk+sj+s, ‖s‖, ∇f's in one pass
    step_names = [f"step_{nm}{sfx}" for nm in ("l1", "l0", "lhalf") for sfx in ("_once", "", "box_vec", "box_scalar")]
    if any(re.search(args.only, nm) for nm in step_names + ["step_l1_once_unfused"]):
        xsy = torch.empty(n, dtype=tdt, device=dev)
        for nm, h in (("l1", sp.NormL1(lam)), ("l0", sp.NormL0(lam)), ("lhalf", sp.RootNormLhalf(lam))):
            once = sp.shifted(h, xk)
            timeit(f"step_{nm}_once", lambda psi=once: sp.step_(y, psi, q, sigma, xsy=xsy), 4 * R,
                   note="ψ shifted once (R2): 2 reads + 2 writes")
            timeit(f"step_{nm}", lambda psi=two(h): sp.step_(y, psi, q, sigma, xsy=xsy), 5 * R)
            timeit(f"step_{nm}box_vec", lambda psi=two(h, l, u): sp.step_(y, psi, q, sigma, xsy=xsy), 7 * R)
            timeit(f"step_{nm}box_scalar", lambda psi=two(h, -1.0, 1.0): sp.step_(y, psi, q, sigma, xsy=xsy), 5 * R)

        def unfused(psi=sp.shifted(sp.NormL1(lam), xk)):  # the same step as separate sweeps (torch for the BLAS-1 parts)
            mq = q * (-sigma)
            sp.prox_(y, psi, mq, sigma)
            v = psi(y)
            torch.add(xk, y, out=xsy)
            return v, float(torch.linalg.vector_norm(y)), float(torch.dot(q, y))
        timeit("step_l1_once_unfused", unfused, 4 * R, note="prox! + ψ(s) + 4 BLAS-1 sweeps, same result")
    # fused step around iprox! (diagonal model: R2DH / TRDH): D + σ, iprox!, ψ(s), xk+sj+s, ‖s‖, ∇f's, sᵀ(D+σ)s in one
    # pass; σ = `sigma`, D = dpos for the unboxed forms (their iprox! asserts d > 0), the C2 mix d for the Box forms
    istep_names = ["istep_l1_once", "istep_l1", "istep_l0box_vec", "istep_l1box_scalar", "istep_l0box_vec_unfused"]
    if any(re.search(args.only, nm) for nm in istep_names):
        xsy = torch.empty(n, dtype=tdt, device=dev)
        once = sp.shifted(sp.NormL1(lam), xk)
        timeit("istep_l1_once", lambda: sp.istep_(y, once, q, dpos, sigma, xsy=xsy), 5 * R,
               note="ψ shifted once: 3 reads + 2 writes")
        timeit("istep_l1", lambda psi=two(sp.NormL1(lam)): sp.istep_(y, psi, q, dpos, sigma, xsy=xsy), 6 * R)
        l0box = two(sp.NormL0(lam), l, u)
        timeit("istep_l0box_vec", lambda: sp.istep_(y, l0box, q, d, sigma, xsy=xsy), 8 * R)
        timeit("istep_l1box_scalar", lambda psi=two(sp.NormL1(lam), -1.0, 1.0): sp.istep_(y, psi, q, d, sigma, xsy=xsy),
               6 * R)

        def iunfused(s=y, out=xsy):  # the same step as separate sweeps (torch for the BLAS-1 parts)
            dd = d + sigma
            sp.iprox_(s, l0box, q, dd)
            v = l0box(s)
            torch.add(xk, sj, out=out)
            out.add_(s)
            return v, float(torch.linalg.vector_norm(s)), float(torch.dot(q, s)), float(torch.dot(dd * s, s))
        if re.search(args.only, "istep_l0box_vec_unfused"):
            y2, xsy2 = torch.empty_like(y), torch.empty_like(y)
            _, r = sp.istep_(y, l0box, q, d, sigma, xsy=xsy)
            r2 = iunfused(y2, xsy2)
            same = torch.equal(y, y2) and torch.equal(xsy, xsy2)
            print(f"istep_l0box_vec vs unfused: s and xsy bit-identical: {same}; scalars {tuple(r)} vs {r2}", flush=True)
            del y2, xsy2
        timeit("istep_l0box_vec_unfused", iunfused, 8 * R,
               note="D+σ, iprox!, ψ(s), xk+sj+s, ‖s‖, ∇f's, sᵀds as separate sweeps, same result")
    # L1B2 (ball active: Δ = half the unconstrained norm)
    if re.search(args.only, "prox_l1b2"):
        psi0 = two(sp.NormL1(lam), 1e30, sp.NormL2(1.0))
        sp.prox_(y, psi0, q, sigma)
        full = float(torch.linalg.vector_norm((y + sj).double()))
        psi = two(sp.NormL1(lam), 0.5 * full, sp.NormL2(1.0))
        sp.prox_(y, psi, q, sigma)
        passes = psi.last_passes
        # bytes actually moved: decision pass 3R, first search pass 3R + 1W (stashes sj + q in y), later search
        # passes 2R, finish 3R + 1W
        nsearch = max(passes - 2, 0)
        timeit("prox_l1b2", lambda: sp.prox_(y, psi, q, sigma), 3 * R + (4 * R if nsearch else 0) + 2 * R * max(nsearch - 1, 0) + 4 * R,
               note=f"{passes - 1} norm passes (3R, 3R+1W, then 2R each) + 1 finish (4R)")
        timeit("prox_l1b2_inactive", lambda: sp.prox_(y, psi0, q, sigma), 7 * R, note="1 norm pass + finish")
    # the ShiftedNormL1B2 step (q plays ∇f, ν = sigma): the one call spx_step_l1b2 against the base-class composition
    # (spx_step_pre, prox! in place with ψ, spx_step_post), ball active, alternated three times: the comparison is what
    # these rows are for.  The composed form takes the in-place prox! route (no stash, no unverified finish), so its s is
    # held to the L1B2 bar of the fused s, which must equal the stand-alone out-of-place prox!'s bit for bit.
    if any(re.search(args.only, nm) for nm in ("step_l1b2", "step_l1b2_composed", "step_l1b2_inactive")):
        nu = sigma
        xsy_l, s2, y2 = torch.empty_like(y), torch.empty_like(y), torch.empty_like(y)
        qn = q * torch.tensor(-nu, dtype=tdt, device=dev)  # fl(-ν∇f)
        psi0 = two(sp.NormL1(lam), 1e30, sp.NormL2(1.0))
        sp.prox_(y, psi0, qn, nu)
        full = float(torch.linalg.vector_norm((y + sj).double()))
        psi = two(sp.NormL1(lam), 0.5 * full, sp.NormL2(1.0))
        sp.prox_(y2, psi, qn, nu)  # the stand-alone out-of-place prox!
        _, r1 = sp.step_(y, psi, q, nu, xsy=xsy_l)
        fused = psi.last_passes
        same = torch.equal(y, y2)
        _, r2 = sp.ShiftedProximableFunction.step_(psi, s2, q, nu, xsy=xsy_l)
        composed = psi.last_passes
        ulps = 64 if R == 8 else 16
        tol = ulps * torch.finfo(tdt).eps * (y.double().abs() + sj.double().abs() + 1)
        within = bool(((s2.double() - y.double()).abs() <= tol).all())
        del tol
        sp.step_(s2, psi0, q, nu, xsy=xsy_l)
        inactive = psi0.last_passes
        print(f"step_l1b2: fused s bit-identical to the out-of-place prox!: {same}; composed s within "
              f"{ulps} ulp of |s| + |sj| + 1: {within}; passes fused {fused}, composed prox! {composed}, inactive "
              f"{inactive}; scalars {tuple(r1)} vs {tuple(r2)}", flush=True)
        del s2, y2, qn
        # bytes per pass: fused -- decision pass 3R (xk, sj, ∇f), first search pass 3R + 1W (stashes mid in s), later
        # passes 2R (xk, mid), finish 4R + 2W (xk, sj, mid, ∇f -> s, xsy; 3R + 2W without a stash);
        # composed -- step_pre 1R + 1W, every norm pass 3R (in place: no stash), finish 3R + 1W, step_post 4R + 1W
        nsearch = fused - 2
        fused_b = 3 * R + (4 * R + 2 * R * (nsearch - 1) + 6 * R if nsearch > 0 else 5 * R)
        composed_b = 2 * R + 3 * R * (composed - 1) + 4 * R + 5 * R
        for _ in range(3):
            timeit("step_l1b2", lambda: sp.step_(y, psi, q, nu, xsy=xsy_l), fused_b,
                   note=f"{fused} passes: {fused - 1} norm passes (3R, 3R+1W, then 2R each) + finish (4R+2W)")
            timeit("step_l1b2_composed", lambda: sp.ShiftedProximableFunction.step_(psi, y, q, nu, xsy=xsy_l),
                   composed_b, note=f"{composed + 2} passes: step_pre (1R+1W), {composed - 1} norm passes (3R) + "
                                    f"finish (3R+1W) in place, step_post (4R+1W)")
        timeit("step_l1b2_inactive", lambda: sp.step_(y, psi0, q, nu, xsy=xsy_l), 8 * R,
               note=f"{inactive} passes: decision pass (3R) + finish (3R+2W)")
        del xsy_l
    # groups of 64 (and ragged)
    for gname in ("g64", "ragged"):
        names = [f"prox_groupl2_{gname}", f"value_groupl2_{gname}", f"prox_groupl2binf_{gname}",
                 "prox_groupl2binf_g64_biglambda", "step_groupl2_g64", "step_groupl2binf_g64",
                 "step_groupl2binf_g64_composed", "step_groupl2binf_g64_biglambda", "step_groupl2_ragged",
                 "step_groupl2_ragged_composed"]
        if not any(re.search(args.only, nm) for nm in names):
            continue
        if gname == "g64":
            ng = n // 64
            offs = torch.arange(0, n + 1, 64, dtype=torch.int64, device=dev)
        else:
            rng = np.random.default_rng(3)
            sizes = np.floor(np.exp(rng.uniform(0, np.log(4097), n // 400))).astype(np.int64).clip(1, 4096)
            cs = np.concatenate([[0], np.cumsum(sizes)])
            cs = cs[cs <= n]
            if cs[-1] != n:
                cs = np.concatenate([cs, [n]])
            offs = torch.from_numpy(cs).to(dev)
            ng = offs.numel() - 1
        lam_g = uni(12, 1.0, 0.5, m=ng)
        h = sp.GroupNormL2(lam_g, None, offsets=offs)
        psi = sp.shifted(sp.shifted(h, xk), sj)
        timeit(f"prox_groupl2_{gname}", lambda psi=psi: sp.prox_(y, psi, q, 0.3), 4 * R, note=f"{ng} groups")
        timeit(f"value_groupl2_{gname}", lambda psi=psi: psi(y), 3 * R)
        if gname == "g64" and re.search(args.only, "step_groupl2_g64"):
            xsy_g = torch.empty_like(y)
            timeit("step_groupl2_g64", lambda psi=psi: sp.step_(y, psi, q, 0.3, xsy=xsy_g), 5 * R,
                   note="spx_step_groupl2: one pass on this layout (groups <= 256); alg. bytes = 3 reads + 2 writes")
            del xsy_g
        # the step on the ragged layout (groups of 1..4096: every size class) against the base-class composition of
        # the same ψ (spx_step_pre, prox! in place with ψ, spx_step_post), alternated three times
        if gname == "ragged" and any(re.search(args.only, nm) for nm in ("step_groupl2_ragged",
                                                                            "step_groupl2_ragged_composed")):
            step_pair("step_groupl2_ragged", psi, 11, f"{ng} groups")
        psib = sp.shifted(sp.shifted(h, xk, 0.5, sp.NormLinf(1.0)), sj)
        timeit(f"prox_groupl2binf_{gname}", lambda psi=psib: sp.prox_(y, psi, q, 0.3), 4 * R, note=f"{ng} groups")
        if gname == "g64":  # σλ_g >> ||sol_g||: the regime of a sparse solution (root next to the pole of c(n) at σλ)
            hb = sp.GroupNormL2(lam_g * 200.0, None, offsets=offs)
            psil = sp.shifted(sp.shifted(hb, xk, 0.5, sp.NormLinf(1.0)), sj)
            timeit("prox_groupl2binf_g64_biglambda", lambda psi=psil: sp.prox_(y, psi, q, 0.3), 4 * R,
                   note="lambda_g x 200")
            # the one-pass step against the base-class composition of the same ψ (spx_step_pre, prox! in place with
            # ψ(s) from its value pass, spx_step_post), alternated three times: the comparison is what these rows are for
            if any(re.search(args.only, nm) for nm in ("step_groupl2binf_g64", "step_groupl2binf_g64_biglambda")):
                xsy_b = torch.empty_like(y)
                s2, xsy2 = torch.empty_like(y), torch.empty_like(y)
                _, r = sp.step_(y, psib, q, 0.3, xsy=xsy_b)
                _, r2 = sp.ShiftedProximableFunction.step_(psib, s2, q, 0.3, xsy=xsy2)
                same = torch.equal(y, s2) and torch.equal(xsy_b, xsy2)
                print(f"step_groupl2binf_g64 vs composed: s and xsy bit-identical: {same}; scalars {tuple(r)} vs "
                      f"{tuple(r2)}", flush=True)
                del s2, xsy2
                for _ in range(3):
                    timeit("step_groupl2binf_g64", lambda: sp.step_(y, psib, q, 0.3, xsy=xsy_b), 5 * R,
                           note="spx_step_groupl2binf: one pass; alg. bytes = 3 reads + 2 writes")
                    timeit("step_groupl2binf_g64_composed",
                           lambda: sp.ShiftedProximableFunction.step_(psib, y, q, 0.3, xsy=xsy_b), 5 * R,
                           note="step_pre, prox! in place + ψ pass, step_post; alg. bytes as above")
                timeit("step_groupl2binf_g64_biglambda", lambda: sp.step_(y, psil, q, 0.3, xsy=xsy_b), 5 * R,
                       note="lambda_g x 200")
                del xsy_b
    # the step on one group spanning the vector (ShiftedGroupNormL2 built from NormL2): norm pass (3R) and scaling
    # pass (3R+2W) against the composition (step_pre 1R+1W, the prox!'s norm pass 3R and scaling pass 3R+1W with ψ,
    # step_post 4R+1W), alternated three times
    if any(re.search(args.only, nm) for nm in ("step_groupl2_one", "step_groupl2_one_composed")):
        step_pair("step_groupl2_one", sp.shifted(sp.shifted(sp.NormL2(lam), xk), sj), 14, "one group")
    # top-r batch: problems of 65536, r = 1024
    if any(re.search(args.only, nm) for nm in ("prox_indballl0_batch", "prox_indballl0binf_batch", "prox_indballl0_single")):
        pn = 65536
        nprob = n // pn
        for binf in (False, True):
            h = sp.IndBallL0(1024)
            psi = (sp.shifted(h, xk, 1.0, sp.NormLinf(1.0), nprob=nprob) if binf else sp.shifted(h, xk, nprob=nprob))
            psi = sp.shifted(psi, sj)
            timeit(f"prox_indballl0{'binf' if binf else ''}_batch", lambda psi=psi: sp.prox_(y, psi, q, 1.0), 4 * R,
                   note=f"{nprob} problems x {pn}, r=1024")
        psi1 = sp.shifted(sp.shifted(sp.IndBallL0(1 << 20), xk), sj)
        timeit("prox_indballl0_single", lambda: sp.prox_(y, psi1, q, 1.0), 4 * R, note="one vector, r=2^20, global path")
    # the top-r step at the C5 shape (problems of 65536, r = 1024; q plays ∇f): the one-pass step
    # (spx_step_indballl0), the base-class composition (spx_step_pre, prox! in place, ψ(s), spx_step_post) and the
    # caller's separate sweeps (q = -ν∇f into its own buffer, the stream prox!, ψ(s), xsy and the two sums as torch ops),
    # alternated three times: the comparison is what these rows are for
    if any(re.search(args.only, nm) for nm in ("step_indballl0_batch", "step_indballl0binf_batch")):
        pn, nu = 65536, 0.3
        nprob = n // pn
        xsy_b = torch.empty_like(y)

        def sweeps(psi, s, xsy, qbuf):
            torch.mul(q, -nu, out=qbuf)
            sp.prox_(s, psi, qbuf, nu)
            val = psi(s)
            torch.add(xk, sj, out=xsy).add_(s)
            return val, torch.dot(s, s).item(), torch.dot(q, s).item()

        for binf in (False, True):
            h = sp.IndBallL0(1024)
            psi = (sp.shifted(h, xk, 1.0, sp.NormLinf(1.0), nprob=nprob) if binf else sp.shifted(h, xk, nprob=nprob))
            psi = sp.shifted(psi, sj)
            tag = f"step_indballl0{'binf' if binf else ''}_batch"
            if not any(re.search(args.only, nm) for nm in (tag, tag + "_composed", tag + "_sweeps")):
                continue
            s2, xsy2, qbuf = torch.empty_like(y), torch.empty_like(y), torch.empty_like(y)
            _, r1 = sp.step_(y, psi, q, nu, xsy=xsy_b)
            _, r2 = sp.ShiftedProximableFunction.step_(psi, s2, q, nu, xsy=xsy2)
            same = torch.equal(y, s2) and torch.equal(xsy_b, xsy2)
            r3 = sweeps(psi, s2, xsy2, qbuf)
            same = same and torch.equal(y, s2) and torch.equal(xsy_b, xsy2)
            print(f"{tag} vs composed vs sweeps: s and xsy bit-identical: {same}; scalars {tuple(r1)} / {tuple(r2)} / "
                  f"(psi {r3[0]}, snorm {r3[1] ** 0.5}, gdots {r3[2]})", flush=True)
            note = f"{nprob} problems x {pn}, r=1024; alg. bytes = 3 reads + 2 writes"
            for _ in range(3):
                timeit(tag, lambda psi=psi: sp.step_(y, psi, q, nu, xsy=xsy_b), 5 * R, note="one pass; " + note)
                timeit(tag + "_composed", lambda psi=psi: sp.ShiftedProximableFunction.step_(psi, y, q, nu, xsy=xsy_b),
                       5 * R, note="step_pre, prox! in place, ψ(s), step_post; " + note)
                timeit(tag + "_sweeps", lambda psi=psi: sweeps(psi, y, xsy_b, qbuf), 5 * R,
                       note="q buffer, stream prox!, ψ(s), torch xsy / dots; " + note)
            del s2, xsy2, qbuf
        del xsy_b
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        json.dump(results, open(args.json, "w"), indent=1)


if __name__ == "__main__":
    main()
