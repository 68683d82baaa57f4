#!/usr/bin/env python
"""bench.py -- throughput of the shifted prox hot path on B200 (contract: see DESIGN.md §Measurement).

Workload = BASELINE.json configs[1] ("C2"): ShiftedNormL0Box prox!, ShiftedRootNormLhalfBox prox! (vector
l/u bounds) and ShiftedNormL0Box iprox! (diagonal d), n = 2^28 Float64 per GPU.  One step = those three
launches over the batch, the first one with ψ(y) fused into its pass (the model decrease a solver reads after
its prox!); on N > 1 GPUs that scalar is all-reduced inside libshiftedprox (ncclAllReduce on the device slot,
spx_comm_*), so every step of the scaling run carries a collective.  `value` = elements/s over all ranks
(3·n prox evaluations per step and rank) with operands resident in HBM; `e2e` = the same through the
host-buffer C-ABI entry point (pinned host vectors, H2D and D2H inside the timed region); `roofline` = the
dominant kernel against the measured HBM peak; `cpu_baseline` = the oracle port (one thread: the reference is
single-threaded) on a bounded sample; `configs` = every configuration of BASELINE.json (C1 ... C5) timed on its
own after the headline step (CUDA events, median of a few launches), sharded over the ranks with their
collectives at N > 1.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the last timed step returned, so that two builds can be compared output for output on
identical inputs: DIR/prox_l0box.npy, prox_lhalfbox.npy, iprox_l0box.npy (Float64; above 2^21 elements a fixed,
seeded sample of up to 2^21 positions, the same in every run; at N > 1 one file per rank with a `_rank<r>` suffix,
each sampling its own shard with 2^21 / N draws) and psi_prox_l0box.npy (the fused ψ(y), all-reduced at N > 1).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "shiftedproximaloperators.jl_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

SEED = 20261018
LAMBDA, SIGMA = 1.0, 0.1
# algorithmic bytes per element (SURVEY.md §8d): Box prox! with vector bounds 6R, Box iprox! 7R
ALG_BYTES = {"prox_l0box": 48, "prox_lhalfbox": 48, "iprox_l0box": 56}
OPS = ("prox_l0box", "prox_lhalfbox", "iprox_l0box")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2n", type=int, default=28)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--config-reps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def kernel_sources_hash() -> str:
    """sha256 over the CUDA sources of libshiftedprox (what an ncu capture under profiles/ was taken from)."""
    import glob
    import hashlib

    h = hashlib.sha256()
    for f in sorted(glob.glob(os.path.join(PKG, "csrc", "*.cu")) + glob.glob(os.path.join(PKG, "csrc", "*.cuh"))):
        h.update(os.path.basename(f).encode())
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


# ------------------------------------------------------------ CPU reference arm ---
def cpu_sample(n: int):
    """The C2 step on n elements through the oracle port (one thread).  Returns seconds per op."""
    import numpy as np

    from oracle import oracle as orc

    xk = orc.uniform(n, 0, np.float64, 4.0, -2.0)
    sj = orc.uniform(n, 1, np.float64, 1.0, -0.5)
    q = orc.uniform(n, 2, np.float64, 4.0, -2.0)
    l = -(0.25 + orc.uniform(n, 3))
    u = 0.25 + orc.uniform(n, 4)
    b = orc.uniform(n, 6)
    d = 0.5 + orc.uniform(n, 5)
    d = np.where(b < 0.1, -d, d)
    d = np.where((b >= 0.1) & (b < 0.2), 0.0, d)
    t = {}
    t0 = time.perf_counter(); orc.prox_box("l0", xk, sj, q, l, u, LAMBDA, SIGMA); t["prox_l0box"] = time.perf_counter() - t0
    t0 = time.perf_counter(); orc.prox_box("lhalf", xk, sj, q, l, u, LAMBDA, SIGMA); t["prox_lhalfbox"] = time.perf_counter() - t0
    t0 = time.perf_counter(); orc.iprox_box("l0", xk, sj, q, d, l, u, LAMBDA); t["iprox_l0box"] = time.perf_counter() - t0
    return t


def cpu_baseline(budget_s: float):
    n = 1 << 20
    t = cpu_sample(n)  # calibration (also warms the oracle build)
    per_elt = sum(t.values()) / n
    n2 = int(min(1 << 26, max(1 << 20, budget_s / max(per_elt, 1e-12))))
    n2 = 1 << (n2.bit_length() - 1)
    t = cpu_sample(n2)
    total = sum(t.values())
    # the "generous CPU bound" of SURVEY.md §8d: the same oracle port on every host core at once (chunks of the sample
    # in a thread pool; ctypes releases the GIL) -- NOT the reference's behaviour (it is single-threaded), reported only
    all_cores = None
    try:
        from concurrent.futures import ThreadPoolExecutor

        cores = len(os.sched_getaffinity(0))
        chunk = max(1 << 18, n2 // cores)
        with ThreadPoolExecutor(cores) as ex:
            per_thread = list(ex.map(lambda _: sum(cpu_sample(chunk).values()), range(cores)))
        all_cores = {"value": 3 * chunk * cores / max(per_thread), "unit": "elements/s", "cores": cores,
                     "note": "oracle port on every host core at once (one chunk of the sample per core, rate = all chunks "
                             "over the slowest core's operator time); the reference itself is single-threaded"}
    except Exception:
        pass
    return {
        "value": 3 * n2 / total, "unit": "elements/s", "cores": 1, "kind": "port", "all_cores": all_cores,
        "sample": f"C2 step (L0Box prox!, LhalfBox prox!, L0Box iprox!) on n=2^{n2.bit_length() - 1} Float64, "
                  f"oracle port g++ -O2 -ffp-contract=off, 1 thread (the reference is single-threaded Julia; "
                  f"`julia` is not in the image), host has {os.cpu_count()} logical cores",
        "seconds": total,
        "per_op_elements_per_s": {k: n2 / v for k, v in t.items()},
    }, total, n2


def cpu_inputs(n: int):
    import numpy as np

    from oracle import oracle as orc

    xk = orc.uniform(n, 0, np.float64, 4.0, -2.0)
    sj = orc.uniform(n, 1, np.float64, 1.0, -0.5)
    q = orc.uniform(n, 2, np.float64, 4.0, -2.0)
    l = -(0.25 + orc.uniform(n, 3))
    u = 0.25 + orc.uniform(n, 4)
    b = orc.uniform(n, 6)
    d = 0.5 + orc.uniform(n, 5)
    d = np.where(b < 0.1, -d, d)
    d = np.where((b >= 0.1) & (b < 0.2), 0.0, d)
    return xk, sj, q, l, u, d


def cpu_step_all_cores(arrs, cores: int, pool) -> float:
    """One C2 step on the sample, every host core working on its own contiguous chunk of the vectors (the reference is
    elementwise on this path, so the chunks are independent; ctypes releases the GIL).  Returns wall seconds."""
    from oracle import oracle as orc

    xk, sj, q, l, u, d = arrs
    n = q.size
    bounds = [(n * c // cores, n * (c + 1) // cores) for c in range(cores)]

    def work(be):
        b, e = be
        sl = slice(b, e)
        orc.prox_box("l0", xk[sl], sj[sl], q[sl], l[sl], u[sl], LAMBDA, SIGMA)
        orc.prox_box("lhalf", xk[sl], sj[sl], q[sl], l[sl], u[sl], LAMBDA, SIGMA)
        orc.iprox_box("l0", xk[sl], sj[sl], q[sl], d[sl], l[sl], u[sl], LAMBDA)

    t0 = time.perf_counter()
    list(pool.map(work, bounds))
    return time.perf_counter() - t0


def run_reference(args, rank):
    """The reference arm: the reference's algorithm for the C2 step (oracle port: `julia` is not in the image) on the
    host, on EVERY core the process may use -- the vectors cut into one contiguous chunk per core -- although the
    reference itself runs this path on one thread; the one-thread rate of the same port is reported next to it."""
    if rank != 0:
        return
    from concurrent.futures import ThreadPoolExecutor

    steps, warm = args.steps, args.warmup
    cores = max(1, len(os.sched_getaffinity(0)))
    # each step = a bounded sample of the workload; keep the whole run within a few minutes
    n = 1 << 20
    t = cpu_sample(n)
    per_elt = sum(t.values()) / n  # one thread
    one_thread = 3 * n / sum(t.values())
    budget = 120.0 / (steps + warm)
    n2 = int(min(1 << 27, max(1 << 20, cores * budget / max(per_elt, 1e-12))))
    n2 = 1 << (n2.bit_length() - 1)
    arrs = cpu_inputs(n2)
    with ThreadPoolExecutor(cores) as pool:
        for _ in range(warm):
            cpu_step_all_cores(arrs, cores, pool)
        t0 = time.perf_counter()
        tot = 0.0
        for _ in range(steps):
            tot += cpu_step_all_cores(arrs, cores, pool)
        wall = time.perf_counter() - t0
    value = 3 * n2 * steps / tot
    line = {
        "impl": "reference", "metric": "prox_elements_per_s", "value": value, "unit": "elements/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": 1e3 * tot / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(28, sample_log2n=n2.bit_length() - 1),
        "cpu_baseline": {"value": value, "unit": "elements/s", "cores": cores, "kind": "port",
                         "one_thread": {"value": one_thread, "unit": "elements/s",
                                        "note": "the reference runs this path on one thread"},
                         "sample": f"each step = the C2 step on n=2^{n2.bit_length() - 1} Float64 (bounded sample), "
                                   f"oracle port (g++ -O2 -ffp-contract=off), one contiguous chunk per core on "
                                   f"{cores} threads, wall clock of the operator calls; host has {os.cpu_count()} "
                                   f"logical cores"},
        "e2e": {"value": value, "unit": "elements/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": wall,
    }
    print(json.dumps(line), flush=True)


def workload_config(log2n, **extra):
    cfg = {
        "workload": f"C2 (BASELINE.json configs[1]): ShiftedNormL0Box prox! + ShiftedRootNormLhalfBox prox! "
                    f"(vector l/u) + ShiftedNormL0Box iprox! (diagonal d), n=2^{log2n} Float64 per GPU, "
                    f"lambda={LAMBDA}, sigma={SIGMA}",
        "n_per_gpu": 1 << log2n,
        "launches_per_step": 3,
        "fused_value": "psi(y) fused into the L0Box prox! pass of every step (want_value); at N > 1 its scalar is "
                       "all-reduced on the device by libshiftedprox (NCCL) before the one D2H copy",
        "alg_bytes_per_element": ALG_BYTES,
        "l2_policy": "operands larger than L2: each of the 7 streamed vectors is n*8 B (2 GiB at 2^28) vs 126 MB L2",
        "sharding": "contiguous shards, one process per GPU; no data-path collective, one scalar all-reduce "
                    "(sum + infeasibility flag) per step for psi(y)",
    }
    cfg.update(extra)
    return cfg


# -------------------------------------------------------------------- clocks ---
class ClockSampler(threading.Thread):
    def __init__(self, index: int, period=0.005):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._halt = threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    NAMES = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
             0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
             0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def poll(self):
        """One sample (SM clock + throttle reasons)."""
        if self.nv is None:
            return
        try:
            self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            for bit, name in self.NAMES.items():
                if r & bit and name != "gpu_idle":
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        while self.nv is not None and not self._halt.is_set():
            self.poll()
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------- GPU arm ---
DUMP_SAMPLE = 1 << 21  # elements per operation over all ranks: 3 x 16 MiB of Float64


def dump_outputs(dirname, outs, psi_val, rank, world):
    """--dump-outputs: the three result vectors of the step (a fixed, seeded sample of positions when larger than
    DUMP_SAMPLE / world) and the fused ψ(y), as .npy files in DIR."""
    import numpy as np
    import torch

    os.makedirs(dirname, exist_ok=True)
    n, m = outs[0].numel(), DUMP_SAMPLE // world
    idx = None
    if n > m:
        idx = np.unique(np.random.default_rng(SEED).integers(0, n, m))
        idx = torch.from_numpy(idx).to(outs[0].device)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, t in zip(OPS, outs):
        a = t if idx is None else t.index_select(0, idx)
        np.save(os.path.join(dirname, f"{name}{suffix}.npy"), a.cpu().numpy())
    if rank == 0:
        np.save(os.path.join(dirname, "psi_prox_l0box.npy"), np.array([psi_val], dtype=np.float64))


def run_ours(args, rank, local_rank, world):
    import torch

    import shiftedprox as sp
    from shiftedprox import _lib as L

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)
    n = 1 << args.log2n
    ctx = sp.context(dev)
    f64 = torch.float64

    def uniform(stream, scale=1.0, shift=0.0, i0=rank * n):
        t = torch.empty(n, dtype=f64, device=dev)
        L.call("spx_fill_uniform_f64", sp.context(dev), C.c_void_p(t.data_ptr()), C.c_int64(n), C.c_int64(i0),
               C.c_uint64(SEED), C.c_uint64(stream), C.c_double(scale), C.c_double(shift))
        return t

    # the shard of rank r is elements [r n, (r+1) n) of the global synthetic vectors
    xk, sj, q = uniform(0, 4.0, -2.0), uniform(1, 1.0, -0.5), uniform(2, 4.0, -2.0)
    l = uniform(3).add_(0.25).neg_()
    u = uniform(4).add_(0.25)
    d = uniform(5).add_(0.5)
    b = uniform(6)
    d = torch.where(b < 0.1, -d, d)
    d = torch.where((b >= 0.1) & (b < 0.2), torch.zeros_like(d), d)
    del b
    y = torch.empty(n, dtype=f64, device=dev)
    psi_l0 = sp.shifted(sp.shifted(sp.NormL0(LAMBDA), xk, l, u), sj)
    psi_lh = sp.shifted(sp.shifted(sp.RootNormLhalf(LAMBDA), xk, l, u), sj)

    from shiftedprox import sharded as shd

    if world > 1:  # collectives inside the library: ncclAllReduce on the device slots, on the context's stream
        shd.comm_init(dev)
        shd.reduce_scalars(True, dev)

    def step(ev=None, outs=(y, y, y)):
        """One C2 step; the three results go to outs (one vector per operation) and the fused ψ(y) is returned."""
        if ev is not None:
            ev[0].record()
        _, psi_val = sp.prox_(outs[0], psi_l0, q, SIGMA, want_value=True)  # fused ψ(y) (+ all-reduce at N > 1)
        if ev is not None:
            ev[1].record()
        sp.prox_(outs[1], psi_lh, q, SIGMA)
        if ev is not None:
            ev[2].record()
        sp.iprox_(outs[2], psi_l0, q, d)
        if ev is not None:
            ev[3].record()
        return psi_val

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    K, W = args.steps, max(3, args.warmup)
    for _ in range(W):
        step()
    barrier()
    # every operation writes all of its output vector either way, so keeping the three results apart for
    # --dump-outputs moves the same bytes as overwriting one vector
    outs = (y, torch.empty_like(y), torch.empty_like(y)) if args.dump_outputs else (y, y, y)
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = sp.launch_count(dev)
    barrier()
    t_start = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    t_start.record()
    for k in range(K):
        psi_val = step(evs[k], outs)
    t_end.record()
    # the K steps are queued and the GPU is still working through them: a few samples from this thread as well (on
    # some boxes the sampler thread gets a single NVML answer during a 140 ms region)
    for _ in range(4):
        sampler.poll()
    barrier()
    launches = sp.launch_count(dev) - launches0
    collectives = shd.comm_info(dev)[2] if world > 1 else 0
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outs, psi_val, rank, world)
    del outs
    ms_total = t_start.elapsed_time(t_end)
    per_op_ms = {op: sum(evs[k][i].elapsed_time(evs[k][i + 1]) for k in range(K)) / K for i, op in enumerate(OPS)}
    if dist is not None:
        tt = torch.tensor([ms_total], dtype=f64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total = float(tt.item())
    ms_step = ms_total / K
    value = world * 3 * n / (ms_step * 1e-3)
    step_bytes = sum(ALG_BYTES[o] for o in OPS) * n

    # roofline of the dominant kernel
    peak, peak_src = measured_peak()
    dom = max(per_op_ms, key=per_op_ms.get)
    achieved = ALG_BYTES[dom] * n / (per_op_ms[dom] * 1e-3) / 1e9
    # DRAM bytes of the dominant kernel from the committed `ncu --set full` capture -- only while the kernel sources
    # are the ones that capture was taken from (profiles/traffic.json records their hash; a stale entry reads null)
    traffic, traffic_note = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        if tj.get("src_sha256") != kernel_sources_hash():
            traffic_note = "profiles/traffic.json was captured from other kernel sources (hash differs): not reported"
        elif dom in tj and tj[dom].get("log2n") == args.log2n:
            traffic = tj[dom]["dram_bytes_per_launch"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                "frac_of_nominal_8000": achieved / 8000.0,
                "per_kernel": {o: {"ms": per_op_ms[o], "GBps": ALG_BYTES[o] * n / (per_op_ms[o] * 1e-3) / 1e9,
                                   "frac": ALG_BYTES[o] * n / (per_op_ms[o] * 1e-3) / 1e9 / peak} for o in OPS}}

    # end-to-end: host (pinned) buffers through spx_box_host_f64
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, sp, L, dev, dist, world, n, (xk, sj, q, d, l, u))

    # every BASELINE.json configuration on its own (frees the C2 operands first)
    configs = None
    if not args.no_configs:
        c2 = {o: dict(roofline["per_kernel"][o], alg_bytes_per_element=ALG_BYTES[o]) for o in OPS}
        del psi_l0, psi_lh, xk, sj, q, l, u, d, y
        torch.cuda.empty_cache()
        configs = run_configs(args, sp, L, shd, dev, dist, world, rank, peak, c2)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu, _, _ = cpu_baseline(args.cpu_seconds)

    if rank == 0:
        line = {
            "metric": "prox_elements_per_s", "value": value, "unit": "elements/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args.log2n),
            "hbm_gbs": world * step_bytes / (ms_step * 1e-3) / 1e9,
            "hbm_frac_of_measured_peak": step_bytes / (ms_step * 1e-3) / 1e9 / peak,
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "collectives_in_timed_region": collectives, "configs": configs, "host_cores": os.cpu_count(),
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        shd.comm_destroy(dev)
        dist.destroy_process_group()


# ------------------------------------------------- every BASELINE.json configuration ---
def run_configs(args, sp, L, shd, dev, dist, world, rank, peak, c2):
    """C1 ... C5 of BASELINE.json, each timed on its own: CUDA events around single calls, 3 warm-ups, median of
    `--config-reps` launches, operands far larger than L2 (C1's n = 10^6 excepted: it is the reference's own
    CPU-sized case and is launch-bound here).  At N > 1 the vector / the groups / the batch of every configuration
    is split over the ranks (`strong`: C3 and C5 keep their total size, as BASELINE.json defines them; the others
    keep the size per GPU), collectives included: ψ(y) all-reduced on the device, the per-pass sums of the L1B2
    search.  Times are the max over ranks."""
    import torch

    f64, f32 = torch.float64, torch.float32
    reps = max(3, args.config_reps)
    shrink = max(0, 28 - args.log2n)  # --log2n below 28 shrinks every configuration alike (smoke runs)

    def uniform(n, stream, dt=f64, scale=1.0, shift=0.0, i0=0):
        t = torch.empty(n, dtype=dt, device=dev)
        suf, ct = ("f64", C.c_double) if dt == f64 else ("f32", C.c_float)
        L.call(f"spx_fill_uniform_{suf}", sp.context(dev), C.c_void_p(t.data_ptr()), C.c_int64(n), C.c_int64(i0),
               C.c_uint64(SEED), C.c_uint64(stream), ct(scale), ct(shift))
        return t

    def timed(fn, burst=1):
        # burst > 1: that many calls between one pair of events (time per call): the host's launch path, which a single
        # call of a 5 us kernel mostly measures, overlaps with the kernels already queued
        for _ in range(3):
            fn()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in ev:
            a.record()
            for _ in range(burst):
                fn()
            b.record()
        torch.cuda.synchronize()
        ts = sorted(a.elapsed_time(b) / burst for a, b in ev)
        ms = ts[len(ts) // 2]
        if dist is not None:
            tt = torch.tensor([ms], dtype=f64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt.item())
        return ms

    def entry(ms, elems_all_ranks, bytes_per_elt, **extra):
        gbs = bytes_per_elt * elems_all_ranks / (ms * 1e-3) / 1e9
        e = {"ms": ms, "elements_per_s": elems_all_ranks / (ms * 1e-3), "alg_bytes_per_element": bytes_per_elt,
             "GBps": gbs, "frac": gbs / (peak * world), "frac_of_nominal_8000": gbs / (8000.0 * world)}
        e.update(extra)
        return e

    out = {"peak_GBps_per_gpu": peak, "n_gpus": world, "timing": f"CUDA events, median of {reps} after 3 warm-ups, max over ranks"}

    # ---- C1: ShiftedNormL1 prox! Float64, sigma = 0.1 (n = 10^6: the reference's CPU case; n = 2^28: the roofline case)
    c1 = {"workload": "ShiftedNormL1 prox! Float64, lambda=1, sigma=0.1, random q/x/s"}
    for name, n in (("n=1e6", 1_000_000), (f"n=2^{28 - shrink}_per_gpu", 1 << (28 - shrink))):
        xk, sj, q = uniform(n, 0, f64, 4.0, -2.0, rank * n), uniform(n, 1, f64, 1.0, -0.5, rank * n), uniform(n, 2, f64, 4.0, -2.0, rank * n)
        y = torch.empty_like(q)
        psi = sp.shifted(sp.shifted(sp.NormL1(1.0), xk), sj)
        c1[name] = entry(timed(lambda: sp.prox_(y, psi, q, SIGMA)), world * n, 32)
        c1[name + "+psi"] = entry(timed(lambda: sp.prox_(y, psi, q, SIGMA, want_value=True)), world * n, 32,
                                  note="psi(y) fused" + (", scalar all-reduced (NCCL)" if world > 1 else ""))
        if n != 1_000_000:  # the solver step around this prox! in one pass (psi shifted once: 2 reads + 2 writes)
            psi1 = sp.shifted(sp.NormL1(1.0), xk)
            xsy = torch.empty_like(q)
            c1[name + " step"] = entry(timed(lambda: sp.step_(y, psi1, q, SIGMA, xsy=xsy)), world * n, 32,
                                       note="fused solver step (spx_step_sep): q = -nu grad, prox!, psi(s), xk + s, |s|, grad's")
            del psi1, xsy
        if n == 1_000_000:  # launch-bound: the same call 32 times back to back (the four vectors, 32 MB, stay in L2)
            c1[name + "_x32_back_to_back"] = entry(timed(lambda: sp.prox_(y, psi, q, SIGMA), burst=32), world * n, 32,
                                                   note="time per call of 32 queued calls; operands L2-resident (32 MB)")
        del xk, sj, q, y, psi
    out["C1"] = c1
    torch.cuda.empty_cache()

    # ---- C2: from the headline step
    out["C2"] = {"workload": "the headline step (see config.workload); per-kernel split by CUDA events inside the timed region",
                 **c2}

    # ---- C3: L1 BInf (= L1Box with ±Delta) and L1B2, Float32, psi(y) all-reduced
    n3_total = 1 << (30 - shrink) if world > 1 else 1 << (29 - shrink)
    n3 = n3_total // world
    i0 = rank * n3
    xk, sj, q = uniform(n3, 0, f32, 4.0, -2.0, i0), uniform(n3, 1, f32, 1.0, -0.5, i0), uniform(n3, 2, f32, 4.0, -2.0, i0)
    y = torch.empty_like(q)
    c3 = {"workload": f"ShiftedNormL1 BInf trust region (L1Box, scalar bounds ±0.75) and ShiftedNormL1B2 (ball active) prox! "
                      f"Float32, n=2^{n3_total.bit_length() - 1} in total over {world} GPU(s), psi(y) fused and all-reduced",
          "n_total": n3_total, "scaling": "strong" if world > 1 else "single GPU (2^30 Float32 x 4 vectors does not leave room for C3 at N=1 next to nothing else: 2^29)"}
    box = sp.shifted(sp.shifted(sp.NormL1(1.0), xk, -0.75, 0.75), sj)
    c3["prox_l1binf"] = entry(timed(lambda: sp.prox_(y, box, q, SIGMA)), n3_total, 16)
    c3["prox_l1binf+psi"] = entry(timed(lambda: sp.prox_(y, box, q, SIGMA, want_value=True)), n3_total, 16,
                                  note="psi(y) fused" + (", scalar all-reduced (NCCL)" if world > 1 else ""))
    pb0 = sp.shifted(sp.shifted(sp.NormL1(1.0), xk, 1.0e9, sp.NormL2(1.0)), sj)
    sp.prox_(y, pb0, q, SIGMA)  # inactive ball: y = ProjB(-xk) - sj
    ss = (sj + y).double().square_().sum()
    if dist is not None:
        dist.all_reduce(ss)
    full = float(ss.sqrt().item())
    del ss
    pb = sp.shifted(sp.shifted(sp.NormL1(1.0), xk, 0.5 * full, sp.NormL2(1.0)), sj)
    ms = timed(lambda: sp.prox_(y, pb, q, SIGMA, want_value=True))
    passes = pb.last_passes
    nsearch = max(passes - 2, 0)
    b_l1b2 = 4 * (3 + (4 if nsearch else 0) + 2 * max(nsearch - 1, 0) + 4)
    c3["prox_l1b2+psi"] = entry(ms, n3_total, b_l1b2, passes=passes,
                                note=f"{passes - 1} norm passes (3R, 3R+1W, then 2R each) + finish (4R); every pass ends in one "
                                     f"all-reduce of its partial sums" if world > 1 else f"{passes - 1} norm passes + finish")
    c3["prox_l1b2+psi"]["frac_single_pass_16B"] = 16 * n3_total / (ms * 1e-3) / 1e9 / (peak * world)
    del xk, sj, q, y, box, pb0, pb
    out["C3"] = c3
    torch.cuda.empty_cache()

    # ---- C4: groups of 64 (10^7 groups) and ragged groups 1..4096, Float64
    ng = (10_000_000 >> shrink)
    n4 = ng * 64
    g0 = rank * ng
    xk, sj, q = uniform(n4, 0, f64, 4.0, -2.0, g0 * 64), uniform(n4, 1, f64, 1.0, -0.5, g0 * 64), uniform(n4, 2, f64, 4.0, -2.0, g0 * 64)
    lam_g = uniform(ng, 12, f64, 1.0, 0.5, g0)
    offs = torch.arange(0, n4 + 1, 64, dtype=torch.int64, device=dev)
    y = torch.empty_like(q)
    h = sp.GroupNormL2(lam_g, None, offsets=offs)
    c4 = {"workload": f"ShiftedGroupNormL2 / ShiftedGroupNormL2Binf prox! Float64, {ng} groups of 64 per GPU (lambda_g = 0.5+u, "
                      f"sigma=0.3, Delta=0.5), plus ragged groups 1..4096 (log-uniform sizes) over the same vector",
          "groups_per_gpu": ng, "scaling": "weak (groups split at group boundaries, no data-path collective)"}
    bpe = 32 + 16.0 / 64
    psi = sp.shifted(sp.shifted(h, xk), sj)
    c4["prox_groupl2_g64"] = entry(timed(lambda: sp.prox_(y, psi, q, 0.3)), world * n4, bpe)
    c4["prox_groupl2_g64+psi"] = entry(timed(lambda: sp.prox_(y, psi, q, 0.3, want_value=True)), world * n4, bpe,
                                       note="psi(y) fused" + (", scalar all-reduced (NCCL)" if world > 1 else ""))
    # the solver step around this prox! (SURVEY.md 8f rank 1): q = -nu grad, prox!, psi(s), xk + sj + s, |s|, grad's in
    # ONE pass on this layout (spx_step_groupl2); q stands in for the gradient
    xsy = torch.empty_like(q)
    c4["step_groupl2_g64"] = entry(timed(lambda: sp.step_(y, psi, q, 0.3, xsy=xsy)), world * n4, 40 + 16.0 / 64,
                                   note="fused solver step: 3 reads + 2 writes, three scalars"
                                        + (" all-reduced on the device" if world > 1 else ""))
    del xsy
    psib = sp.shifted(sp.shifted(h, xk, 0.5, sp.NormLinf(1.0)), sj)
    c4["prox_groupl2binf_g64"] = entry(timed(lambda: sp.prox_(y, psib, q, 0.3)), world * n4, bpe)
    import numpy as np

    rng = np.random.default_rng(3)
    sizes = np.floor(np.exp(rng.uniform(0, np.log(4097), n4 // 400))).astype(np.int64).clip(1, 4096)
    cs = np.concatenate([[0], np.cumsum(sizes)])
    cs = cs[cs <= n4]
    if cs[-1] != n4:
        cs = np.concatenate([cs, [n4]])
    offs_r = torch.from_numpy(cs).to(dev)
    ngr = offs_r.numel() - 1
    lam_r = uniform(ngr, 12, f64, 1.0, 0.5, 0)
    hr = sp.GroupNormL2(lam_r, None, offsets=offs_r)
    bper = 32 + 16.0 * ngr / n4
    psi = sp.shifted(sp.shifted(hr, xk), sj)
    c4["prox_groupl2_ragged"] = entry(timed(lambda: sp.prox_(y, psi, q, 0.3)), world * n4, bper, groups_per_gpu=ngr)
    psib = sp.shifted(sp.shifted(hr, xk, 0.5, sp.NormLinf(1.0)), sj)
    c4["prox_groupl2binf_ragged"] = entry(timed(lambda: sp.prox_(y, psib, q, 0.3)), world * n4, bper, groups_per_gpu=ngr)
    del xk, sj, q, y, psi, psib, h, hr, offs, offs_r, lam_g, lam_r
    out["C4"] = c4
    torch.cuda.empty_cache()

    # ---- C5: top-r batch, 4096 problems of 65536, r = 1024, Float64; the batch is split over the ranks
    nprob_total = max(world, 4096 >> shrink)
    lo, hi = shd.shard_problems(nprob_total, world, rank)
    npr, pn = hi - lo, 65536
    n5 = npr * pn
    xk, sj, q = uniform(n5, 0, f64, 4.0, -2.0, lo * pn), uniform(n5, 1, f64, 1.0, -0.5, lo * pn), uniform(n5, 2, f64, 4.0, -2.0, lo * pn)
    y = torch.empty_like(q)
    c5 = {"workload": f"ShiftedIndBallL0BInf / ShiftedIndBallL0 prox! Float64, batch of {nprob_total} independent problems of "
                      f"n=65536, r=1024, Delta=1, split over {world} GPU(s) ({npr} problems on rank 0)",
          "scaling": "strong (the batch keeps its size)" if world > 1 else "single GPU"}
    hb = sp.IndBallL0(1024)
    psi = sp.shifted(sp.shifted(hb, xk, 1.0, sp.NormLinf(1.0), nprob=npr), sj)
    c5["prox_indballl0binf_batch"] = entry(timed(lambda: sp.prox_(y, psi, q, 1.0)), nprob_total * pn, 32)
    psi = sp.shifted(sp.shifted(hb, xk, nprob=npr), sj)
    c5["prox_indballl0_batch"] = entry(timed(lambda: sp.prox_(y, psi, q, 1.0)), nprob_total * pn, 32)
    del xk, sj, q, y, psi
    out["C5"] = c5
    torch.cuda.empty_cache()
    return out


def run_e2e(args, sp, L, dev, dist, world, n, dev_inputs):
    import torch

    f64 = torch.float64
    xk, sj, q, d, l, u = dev_inputs
    from shiftedprox import hostpath as hp

    # N > 1: keep each rank's host buffers (first touch) and its copy threads on the cores next to its GPU --
    # NVML's CPU affinity of the device when available, else an even split of the cores by local rank
    affinity = None
    if world > 1:
        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(dev.index)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
            cores = [64 * w + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1]
            allowed = sorted(set(cores) & set(os.sched_getaffinity(0)))
            if allowed:
                os.sched_setaffinity(0, allowed)
                affinity = f"nvml ({len(allowed)} cores)"
        except Exception:
            try:
                cores = sorted(os.sched_getaffinity(0))
                per = max(1, len(cores) // world)
                mine = cores[dev.index * per:(dev.index + 1) * per] or cores
                os.sched_setaffinity(0, mine)
                affinity = f"even split ({len(mine)} cores)"
            except Exception:
                affinity = None
    try:
        host = [torch.empty(n, dtype=f64, pin_memory=True) for _ in range(9)]
    except Exception as e:  # not enough lockable host memory
        return {"value": None, "unit": "elements/s", "error": f"pinned allocation failed: {e}"}
    hxk, hsj, hq, hd, hl, hu, hy0, hy1, hy2 = host
    for h, t in zip((hxk, hsj, hq, hd, hl, hu), (xk, sj, q, d, l, u)):
        h.copy_(t)
    torch.cuda.synchronize()
    ctx = sp.context(dev)
    # the C2 step at one shifted point: every input vector (xk, sj, q, d, l, u) crosses PCIe once per step,
    # the three results travel back
    jobs = [dict(op="l0", y=hy0, q=hq, lam=LAMBDA, sigma=SIGMA), dict(op="lhalf", y=hy1, q=hq, lam=LAMBDA, sigma=SIGMA),
            dict(op="l0", y=hy2, q=hq, d=hd, lam=LAMBDA)]

    def host_step():
        hp.box_multi_host(ctx, jobs, hxk, hsj, hl, hu, chunk=1 << 22)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    host_step()  # warm-up (allocates the staging ring)
    K = max(1, args.e2e_steps)
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        host_step()
    barrier()
    dt = time.perf_counter() - t0
    if dist is not None:
        tt = torch.tensor([dt], dtype=f64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
    h2d = 6 * n * 8  # xk, sj, q (= g), d, l, u
    d2h = 3 * n * 8  # one result per operation
    # what ONE drop-in prox!(y::Vector, ψ, q, σ) on host vectors costs (spx_box_host_f64: ShiftedNormL0Box prox!, five
    # input vectors up, one result down) -- the reference API has no multi-operation verb
    def single_op():
        hp.box_host(ctx, "l0", hy0, hxk, hsj, hq, hl, hu, LAMBDA, SIGMA, chunk=1 << 22)

    single_op()
    barrier()
    t1 = time.perf_counter()
    for _ in range(K):
        single_op()
    barrier()
    dt1 = time.perf_counter() - t1
    if dist is not None:
        tt = torch.tensor([dt1], dtype=f64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt1 = float(tt.item())
    single = {"api": "spx_box_host_f64: one ShiftedNormL0Box prox! on pinned host vectors", "ms_per_call": 1e3 * dt1 / K,
              "elements_per_s": world * n * K / dt1, "h2d_bytes_per_call": 5 * n * 8, "d2h_bytes_per_call": n * 8,
              "pcie_gbs_per_gpu": 6 * n * 8 * K / dt1 / 1e9}
    return {"value": world * 3 * n * K / dt, "unit": "elements/s", "h2d_bytes_per_step": h2d, "single_op": single,
            "pcie_gbs_per_gpu": (h2d + d2h) * K / dt / 1e9,
            "d2h_bytes_per_step": d2h, "steps": K, "ms_per_step": 1e3 * dt / K,
            "pcie_gbs": (h2d + d2h) * K / dt / 1e9,
            "api": "spx_box_multi_host_f64: the three operations of the step at one shifted point, pinned host vectors, "
                   "4 Mi-element chunks, 3-stream H2D/kernel/D2H pipeline, every input vector uploaded once per step",
            "host_affinity": affinity}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
