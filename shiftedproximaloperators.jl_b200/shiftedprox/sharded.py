"""Host-side logic for one vector (or one batch) sharded over the GPUs of a box, one process per GPU.

Nothing here touches the data path: elementwise / Box / group / batched top-r proxes run on each rank's
contiguous shard with no collective (SURVEY.md §8e).  Collectives exist only where the path has a real
exchange: the scalar ψ(y) (sum + infeasibility flag) and the K partial sums per pass of the ℓ2 trust-region
root search (ShiftedNormL1B2).

Two ways to run them:

* `comm_init()` + `reduce_scalars(True)`: the collectives run INSIDE libshiftedprox -- ncclAllReduce over NVLink on
  the context's stream, directly on the device slots the kernels fold into, before the one D2H copy of the call.
  Every verb of the host mirror (`ψ(y)`, `prox_(..., want_value=True)`, `step_`, ShiftedNormL1B2's `prox_`) then
  returns whole-vector scalars, identical on every rank, with no host staging.  `torch.distributed` only carries
  the 128-byte NCCL id to the ranks.
* the callback forms below (`value_sharded`, `prox_l1b2_sharded_`, ...): the host all-reduces through
  `torch.distributed` (gloo in the CPU tests, NCCL on GPUs).  Kept as the fallback and for the CPU tests.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist


# ------------------------------------------------- collectives inside the library ---
def comm_init(device=None, group=None, peer=None) -> None:
    """Attach an NCCL communicator to this rank's libshiftedprox context (spx_comm_init): rank 0 draws the id
    (spx_comm_unique_id), `torch.distributed` broadcasts its 128 bytes, every rank joins.

    `peer` (default: on unless SPX_PEER=0): also map every rank's exchange buffer into every process
    (spx_comm_peer_export / _attach, CUDA IPC over NVLink), so that the scalar reductions are finished by the fold
    kernel itself instead of a separate NCCL launch.  All ranks agree on the outcome: if one cannot map a peer
    (no P2P path, IPC closed in the container) every rank detaches and the reductions stay on NCCL."""
    import os

    from . import _lib as L, context

    if not (dist.is_available() and dist.is_initialized()):
        raise RuntimeError("comm_init needs an initialised torch.distributed process group (to pass the NCCL id)")
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    ctx = context(dev)
    idbuf = (C.c_ubyte * 128)()
    if rank == 0:
        L.call("spx_comm_unique_id", idbuf)
    carrier = dev if dist.get_backend(group) == "nccl" else torch.device("cpu")
    t = torch.tensor(list(idbuf), dtype=torch.uint8, device=carrier)
    dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    raw = bytes(t.cpu().tolist())
    L.call("spx_comm_init", ctx, C.c_int32(world), C.c_int32(rank), C.c_char_p(raw))
    if peer is None:
        peer = os.environ.get("SPX_PEER", "1") != "0"
    if peer and 1 < world <= 16:
        _peer_attach(ctx, rank, world, carrier, group)


def _peer_attach(ctx, rank, world, carrier, group) -> bool:
    from . import _lib as L

    hbuf = (C.c_ubyte * 64)()
    ok = 1
    try:
        L.call("spx_comm_peer_export", ctx, hbuf)
    except Exception:
        ok = 0
    mine = torch.tensor(list(hbuf), dtype=torch.uint8, device=carrier)
    every = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(every, mine, group=group)
    if ok:
        raw = b"".join(bytes(e.cpu().tolist()) for e in every)
        try:
            L.call("spx_comm_peer_attach", ctx, C.c_int32(world), C.c_int32(rank), C.c_char_p(raw))
        except Exception:
            ok = 0
    flag = torch.tensor([ok], dtype=torch.int32, device=carrier)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
    if int(flag.item()) == 0:
        L.call("spx_comm_peer_detach", ctx)
        return False
    return True


def comm_peer_active(device=None) -> bool:
    """True when this rank's scalar reductions go over the peer-mapped exchange buffers (one fused kernel)."""
    from . import _lib as L, context

    lib = L.lib()
    lib.spx_comm_peer_active.restype = C.c_int32
    return bool(lib.spx_comm_peer_active(context(device if device is not None else torch.cuda.current_device())))


def comm_destroy(device=None) -> None:
    from . import _lib as L, context

    L.call("spx_comm_destroy", context(device if device is not None else torch.cuda.current_device()))


def reduce_scalars(on: bool, device=None) -> None:
    """spx_comm_reduce_scalars: with `on`, every scalar the library hands back is the whole-vector value (all-reduced
    on the device); every rank must then make the same calls in the same order."""
    from . import _lib as L, context

    L.call("spx_comm_reduce_scalars", context(device if device is not None else torch.cuda.current_device()),
           C.c_int32(1 if on else 0))


def comm_info(device=None):
    """(nranks, rank, collectives issued so far) of this rank's context."""
    from . import _lib as L, context

    a, b, c = C.c_int32(), C.c_int32(), C.c_int64()
    L.call("spx_comm_info", context(device if device is not None else torch.cuda.current_device()), C.byref(a),
           C.byref(b), C.byref(c))
    return a.value, b.value, c.value


# ------------------------------------------------------------------ partitioning ---
def shard_bounds(n: int, world: int, rank: int, align: int = 4) -> Tuple[int, int]:
    """Contiguous shard [lo, hi) of rank `rank`; interior boundaries are multiples of `align` elements so that
    every shard base stays 16-byte aligned (align=4 covers Float32; 2 suffices for Float64)."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError("bad world/rank")
    per = -(-n // world)
    per = -(-per // align) * align
    lo = min(n, rank * per)
    hi = min(n, lo + per)
    return lo, hi


def shard_groups(offsets: Sequence[int], world: int) -> List[Tuple[int, int]]:
    """Split groups (CSR offsets) at group boundaries into `world` contiguous runs balancing the number of
    elements.  Returns [(g_lo, g_hi)] per rank (possibly empty runs at the end)."""
    offs = np.asarray(offsets, dtype=np.int64)
    ng = offs.size - 1
    n = int(offs[-1])
    cuts = [0]
    for r in range(1, world):
        target = n * r // world
        g = int(np.searchsorted(offs, target, side="left"))
        g = max(cuts[-1], min(ng, g))
        cuts.append(g)
    cuts.append(ng)
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def shard_problems(nprob: int, world: int, rank: int) -> Tuple[int, int]:
    """Batch of independent problems (top-r): problems [lo, hi) of rank `rank`."""
    per = -(-nprob // world)
    lo = min(nprob, rank * per)
    return lo, min(nprob, lo + per)


# ----------------------------------------------------------------------- ψ(y) ---
def combine_value(kind: str, partial_sum: float, infeasible: float, lam: float, dtype, r: int = 0) -> float:
    """Turn the all-reduced (Σ, infeasible-flag) into ψ(y): λ·Σ rounded like the reference's value functor
    (in R), count ≤ r ? 0 : Inf for IndBallL0, Inf if any shard was infeasible."""
    if infeasible > 0:
        return math.inf
    if kind == "indballl0":
        return 0.0 if partial_sum <= r else math.inf
    rt = np.float64 if dtype in (torch.float64, np.float64) else np.float32
    return float(rt(lam) * rt(partial_sum))


def allreduce_value(kind: str, local_sum: float, local_infeasible: bool, lam: float, dtype, r: int = 0,
                    device=None, group=None) -> float:
    """Scalar all-reduce of ψ(y) partials: SUM for Σ, MAX for the infeasibility flag (so `Inf` survives as a
    flag, never as Inf - Inf)."""
    t = torch.tensor([local_sum, 1.0 if local_infeasible else 0.0], dtype=torch.float64, device=device or "cpu")
    if dist.is_available() and dist.is_initialized():
        s = t[:1].clone()
        f = t[1:].clone()
        dist.all_reduce(s, op=dist.ReduceOp.SUM, group=group)
        dist.all_reduce(f, op=dist.ReduceOp.MAX, group=group)
        t = torch.cat([s, f])
    return combine_value(kind, float(t[0]), float(t[1]), lam, dtype, r)


_KIND = {"l1": 0, "l0": 1, "lhalf": 2, "indballl0": 3}


def value_sharded(psi, y_local: torch.Tensor, group=None) -> float:
    """ψ(y) of a separable / Box ψ whose vectors are this rank's shard (GPU path)."""
    from . import _lib as L, _BoxBase, _p  # local import: needs the CUDA library

    kind = {L.H_L1: "l1", L.H_L0: "l0", L.H_LHALF: "lhalf", L.H_INDBALLL0: "indballl0"}[psi._H_KIND]
    out = (C.c_double * 2)()
    boxed = isinstance(psi, _BoxBase)
    if boxed:
        lb, ub = psi._bounds()
        psi._call("value_partial", C.c_int32(psi._H_KIND), C.c_int64(psi.n), _p(psi.xk), _p(psi.sj), _p(y_local),
                  C.byref(lb), C.byref(ub), psi._sel.ref(), C.c_int32(1), out)
    else:
        psi._call("value_partial", C.c_int32(psi._H_KIND), C.c_int64(psi.n), _p(psi.xk), _p(psi.sj), _p(y_local),
                  None, None, None, C.c_int32(0), out)
    return allreduce_value(kind, out[0], out[1] > 0, getattr(psi.h, "lam", 0.0), psi.xk.dtype,
                           getattr(psi.h, "r", 0), device=psi.xk.device, group=group)


# ------------------------------------------------------- fused solver step, sharded ---
def allreduce_step(psi_value: float, s_sumsq: float, gdots: float, device=None, group=None):
    """Scalars of a fused solver step over all shards: (ψ(s), ‖s‖₂, ∇f's) from the per-shard
    (ψ(s_shard), Σs², Σ∇f·s) -- one SUM all-reduce of three doubles.  ψ is a sum over entries for every separable
    h and an infeasible shard contributes Inf, which survives the sum (ψ >= 0: never Inf - Inf)."""
    t = torch.tensor([psi_value, s_sumsq, gdots], dtype=torch.float64, device=device or "cpu")
    if dist.is_available() and dist.is_initialized():
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    v = t.tolist()
    return v[0], math.sqrt(v[1]), v[2]


def step_sharded_(s_local, psi, grad_local, nu, xsy_local=None, group=None):
    """Fused solver step (shiftedprox.step_) on this rank's contiguous shard: no data-path collective, one scalar
    all-reduce.  Returns (s_local, StepResult) with the whole-vector scalars, identical on every rank."""
    from . import StepResult  # local import: needs the CUDA library

    _, r = psi.step_(s_local, grad_local, nu, xsy_local)
    return s_local, StepResult(*allreduce_step(r.psi, r.snorm * r.snorm, r.gdots, device=s_local.device, group=group))


# ------------------------------------------------------- the all-reduce callback ---
_REDUCE_BUFS: dict = {}


def _make_reduce(dev, group):
    """SUM all-reduce of `count` doubles handed over by libshiftedprox (spx_allreduce_sum_fn): a pinned host
    mirror and a device buffer are kept per device, the values travel H2D -> NCCL -> D2H on the current stream."""

    def _reduce(_user, vals, count):
        # Never let an exception cross the C boundary, and never leave the peers alone in the collective: whatever
        # fails locally, this rank still joins the all-reduce (with a poisoned status word riding along), so every
        # rank sees the failure and aborts together instead of one returning early and the others hanging.
        status = 0.0
        host = buf = None
        try:
            key = (dev.index, max(count + 1, 64))
            bufs = _REDUCE_BUFS.get(key)
            if bufs is None:
                h = torch.empty(max(count + 1, 64), dtype=torch.float64, pin_memory=dev.type == "cuda")
                bufs = _REDUCE_BUFS[key] = (h, torch.empty(max(count + 1, 64), dtype=torch.float64, device=dev))
            host, buf = bufs
            src = np.ctypeslib.as_array(vals, shape=(count,))
            host[:count].numpy()[:] = src  # bulk copy, no per-element Python loop
        except Exception:
            status = 1.0
        try:
            if host is None:
                host = torch.zeros(count + 1, dtype=torch.float64)
                buf = torch.zeros(count + 1, dtype=torch.float64, device=dev)
            host[count] = status
            buf[:count + 1].copy_(host[:count + 1], non_blocking=True)
            dist.all_reduce(buf[:count + 1], op=dist.ReduceOp.SUM, group=group)
            host[:count + 1].copy_(buf[:count + 1], non_blocking=True)
            if dev.type == "cuda":
                torch.cuda.current_stream(dev).synchronize()
            if float(host[count]) != 0.0:
                return -1  # some rank failed: every rank returns the error
            np.ctypeslib.as_array(vals, shape=(count,))[:] = host[:count].numpy()
            return 0
        except Exception:
            return -1

    return _reduce


# ---------------------------------------------------------------- L1B2 sharded ---
def prox_l1b2_sharded_(y_local, psi, q_local, sigma, group=None, want_value=False):
    """ShiftedNormL1B2 prox! on a sharded vector: every pass's K partial sums of squares go through one
    all-reduce (SUM, Float64); the scalar root search runs replicated inside libshiftedprox."""
    from . import _lib as L, _p

    dev = psi.xk.device

    cb = L.ALLREDUCE_FN(_make_reduce(dev, group))
    passes = C.c_int32()
    out = C.c_double() if want_value else None
    psi._call("prox_l1b2_sharded", C.c_int64(psi.n), _p(y_local), _p(psi.xk), _p(psi.sj), _p(q_local),
              C.c_double(psi.h.lam), C.c_double(sigma), C.c_double(psi.Delta), C.c_double(psi.chi.lam), cb, None,
              C.byref(passes), C.byref(out) if want_value else None)
    psi.last_passes = passes.value
    return (y_local, out.value) if want_value else y_local


def step_l1b2_sharded_(s_local, psi, grad_local, nu, xsy_local=None, group=None):
    """ShiftedNormL1B2 solver step (ShiftedNormL1B2.step_) on a sharded vector: the search's partial sums go through
    one all-reduce per pass, the finish's four sums (ψ's two, Σs², Σ∇f·s) through one more.  Returns
    (s_local, StepResult) with the whole-vector scalars, identical on every rank."""
    from . import _lib as L, StepResult

    cb = L.ALLREDUCE_FN(_make_reduce(psi.xk.device, group))
    out, passes = (C.c_double * 3)(), C.c_int32()
    psi._call("step_l1b2_sharded", *psi._step_args(s_local, grad_local, nu, xsy_local), cb, None, C.byref(passes), out)
    psi.last_passes = passes.value
    return s_local, StepResult(out[0], math.sqrt(out[1]), out[2])


# ----------------------------------------------------- single-vector top-r sharded ---
def prox_indballl0_sharded_(y_local, psi, q_local, n_global: int, group=None):
    """ShiftedIndBallL0(BInf) prox! of ONE vector spread over the ranks in rank order (this rank holds
    psi.n contiguous elements): each radix digit's 2048-bin histogram is all-reduced (SUM), every rank picks
    the same digit, and ties at the threshold go to the lowest global index (SURVEY.md §8e)."""
    from . import _lib as L, _p, ShiftedIndBallL0BInf

    dev = psi.xk.device
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1

    binf = isinstance(psi, ShiftedIndBallL0BInf)
    # a communicator on the context (comm_init): histograms and tie counts are all-reduced on the device (NULL callback)
    in_library = world > 1 and comm_info(dev)[0] == world
    if in_library:
        cb = C.cast(None, L.ALLREDUCE_FN)
    elif world > 1:
        cb = L.ALLREDUCE_FN(_make_reduce(dev, group))
    else:
        cb = L.ALLREDUCE_FN(lambda u, v, c: 0)
    psi._call("prox_indballl0_sharded", C.c_int64(psi.n), C.c_int64(n_global), _p(y_local), _p(psi.xk), _p(psi.sj),
              _p(q_local), C.c_int64(psi.h.r), C.c_int32(1 if binf else 0),
              C.c_double(psi.Delta if binf else 0.0), C.c_int32(rank), C.c_int32(world), cb, None)
    return y_local
