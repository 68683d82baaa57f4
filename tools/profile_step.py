#!/usr/bin/env python
"""torch.profiler kernel list of the C2 step that bench.py times (L0Box prox! with fused ψ, LhalfBox prox!, L0Box
iprox!, vector bounds, Float64), on the same seeded operands.

    python tools/profile_step.py [--log2n 28] [--steps 3] [--out FILE]

Prints (and writes to FILE) every device activity of the profiled steps in launch order with its duration and the
idle gap before it, then the per-kernel totals.  The gap after the fused-ψ call is the host round trip that returns ψ.
"""
import argparse
import ctypes as C
import os
import sys

import torch
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "shiftedproximaloperators.jl_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
import bench  # noqa: E402  (SEED, LAMBDA, SIGMA of the timed workload)
import shiftedprox as sp  # noqa: E402
from shiftedprox import _lib as L  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", type=int, default=28)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = 0
    n = 1 << args.log2n

    def uniform(stream, scale=1.0, shift=0.0):
        t = torch.empty(n, dtype=torch.float64, device=dev)
        L.call("spx_fill_uniform_f64", sp.context(dev), C.c_void_p(t.data_ptr()), C.c_int64(n), C.c_int64(0),
               C.c_uint64(bench.SEED), C.c_uint64(stream), C.c_double(scale), C.c_double(shift))
        return t

    xk, sj, q = uniform(0, 4.0, -2.0), uniform(1, 1.0, -0.5), uniform(2, 4.0, -2.0)
    lo, up = uniform(3).add_(0.25).neg_(), uniform(4).add_(0.25)
    d = uniform(5).add_(0.5)
    b = uniform(6)
    d = torch.where(b < 0.1, -d, d)
    d = torch.where((b >= 0.1) & (b < 0.2), torch.zeros_like(d), d)
    del b
    y = torch.empty(n, dtype=torch.float64, device=dev)
    psi_l0 = sp.shifted(sp.shifted(sp.NormL0(bench.LAMBDA), xk, lo, up), sj)
    psi_lh = sp.shifted(sp.shifted(sp.RootNormLhalf(bench.LAMBDA), xk, lo, up), sj)

    def step():
        sp.prox_(y, psi_l0, q, bench.SIGMA, want_value=True)
        sp.prox_(y, psi_lh, q, bench.SIGMA)
        sp.iprox_(y, psi_l0, q, d)

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            step()
        torch.cuda.synchronize()
    evs = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                 key=lambda e: e.time_range.start)
    props = torch.cuda.get_device_properties(dev)
    lines = [f"# {props.name}, n = 2^{args.log2n} Float64, {args.steps} steps; times in us (gap = idle before)"]
    prev_end = None
    for e in evs:
        gap = "" if prev_end is None else f"{e.time_range.start - prev_end:10.1f}"
        lines.append(f"{e.time_range.elapsed_us():10.1f} {gap:>10s}  {e.name}")
        prev_end = e.time_range.end
    lines.append("")
    lines.append(prof.key_averages().table(sort_by="cuda_time_total", row_limit=20))
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
