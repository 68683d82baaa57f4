"""shiftedprox -- host-side mirror of the ShiftedProximalOperators.jl API on B200 buffers.

The reference's public verbs (src/ShiftedProximalOperators.jl:11-12) keep their names and
argument meaning; Julia's `!` becomes a trailing underscore:

    shifted(h, x) / shifted(h, x, l, u[, selected]) / shifted(h, x, Δ, χ[, selected]) / shifted(ψ, s)
    shift_(ψ, v)            shift!        ShiftedProximalOperators.jl:72-79
    set_radius_(ψ, Δ)       set_radius!   :93-99
    set_bounds_(ψ, l, u)    set_bounds!   :107-111
    prox_(y, ψ, q, σ)       prox!         per-type methods, see each class
    prox(ψ, q, σ)           prox          :189-190  (writes ψ.sol)
    iprox_(y, ψ, g, d)      iprox!
    iprox(ψ, g, d)          iprox         :180
    ψ(y)                    value         :51-54 and the per-type overrides

Vectors are 1-D contiguous CUDA torch tensors (Float64 or Float32): torch is only the
owner of device memory and streams here.  Every verb is one call into libshiftedprox.so
through the C ABI of include/shiftedprox.h; nothing is computed in Python or on the CPU.
The Julia glue a maintainer would use instead of this module is in
../julia/ShiftedProxB200.jl and INTEGRATION.md.

Indices are 0-based on this side (`selected=range(0, n, 2)` is Julia's `1:2:n`).
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional, Sequence

import torch

from . import _lib as L
from ._lib import SpxError  # noqa: F401

__all__ = [
    "NormL1", "NormL0", "RootNormLhalf", "NormL2", "NormLinf", "GroupNormL2", "IndBallL0",
    "ShiftedProximableFunction", "ShiftedNormL1", "ShiftedNormL0", "ShiftedRootNormLhalf", "ShiftedNormL1Box",
    "ShiftedNormL0Box", "ShiftedRootNormLhalfBox", "ShiftedNormL1B2", "ShiftedIndBallL0", "ShiftedIndBallL0BInf",
    "ShiftedGroupNormL2", "ShiftedGroupNormL2Binf",
    "shifted", "shift_", "set_radius_", "set_bounds_", "prox_", "prox", "iprox_", "iprox", "prox_zero",
    "iprox_zero", "step_", "StepResult", "istep_", "IStepResult", "context", "launch_count",
]

_SUF = {torch.float64: "f64", torch.float32: "f32"}
_CT = {torch.float64: C.c_double, torch.float32: C.c_float}
_BOX_OP = {"l1box": L.BOX_L1, "l0box": L.BOX_L0, "lhalfbox": L.BOX_LHALF}


# ------------------------------------------------------------------ context ---
class _Ctx:
    def __init__(self, device: int):
        self.device = device
        self.handle = C.c_void_p()
        stream = torch.cuda.current_stream(device).cuda_stream
        L.call("spx_ctx_create", C.byref(self.handle), C.c_int32(device), C.c_void_p(stream), C.c_int32(0))
        self.stream = stream

    def use_current_stream(self):
        s = torch.cuda.current_stream(self.device).cuda_stream
        if s != self.stream:
            L.call("spx_ctx_set_stream", self.handle, C.c_void_p(s))
            self.stream = s
        return self.handle


_contexts: dict = {}


def context(device) -> C.c_void_p:
    """spx_ctx of a CUDA device, bound to torch's current stream on it."""
    idx = torch.device(device).index if not isinstance(device, int) else device
    if idx is None:
        idx = torch.cuda.current_device()
    c = _contexts.get(idx)
    if c is None:
        if not torch.cuda.is_available():
            raise RuntimeError("shiftedprox needs a CUDA device (sm_100a); there is no CPU fallback")
        c = _contexts[idx] = _Ctx(idx)
    return c.use_current_stream()


def launch_count(device=None) -> int:
    out = C.c_int64()
    L.call("spx_ctx_launch_count", context(device if device is not None else torch.cuda.current_device()), C.byref(out))
    return out.value


def _vec(t: torch.Tensor, like: Optional[torch.Tensor] = None, name: str = "vector") -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError(f"{name}: expected a CUDA torch tensor (device buffers are owned by the host code)")
    if t.dtype not in _SUF:
        raise TypeError(f"{name}: element type must be float64 or float32, got {t.dtype}")
    if t.dim() != 1 or not t.is_contiguous():
        raise ValueError(f"{name}: expected a contiguous 1-D vector")
    if like is not None:
        if t.dtype != like.dtype:
            raise TypeError(f"{name}: element type {t.dtype} differs from {like.dtype}")
        if t.numel() != like.numel():
            raise ValueError(f"{name}: length {t.numel()} differs from {like.numel()}")
        if t.device != like.device:
            raise ValueError(f"{name}: on {t.device}, expected {like.device}")
    return t


def _copy_strided(dst: torch.Tensor, src: torch.Tensor) -> None:
    L.call("spx_copy_strided", context(dst.device), C.c_int64(dst.numel()), C.c_int32(dst.element_size()),
           C.c_void_p(dst.data_ptr()), C.c_int64(dst.stride(0)), C.c_void_p(src.data_ptr()), C.c_int64(src.stride(0)))


def _adopt(t: torch.Tensor, like: Optional[torch.Tensor] = None, name: str = "vector") -> torch.Tensor:
    """A shift vector: contiguous (aliased as is, like the reference), or a strided 1-D view -- the reference's
    `SubArray` shifts (`x = view(y, 1:2:10); shifted(h, x)`, test/runtests.jl:199-200).  The kernels stream
    contiguous operands, so a strided view gets a contiguous shadow that is re-gathered from the view before every
    call (the caller may have written the parent array) and scattered back when shift! writes it."""
    if isinstance(t, torch.Tensor) and t.is_cuda and t.dim() == 1 and not t.is_contiguous() and t.dtype in _SUF \
            and t.stride(0) != 0:
        shadow = torch.empty(t.numel(), dtype=t.dtype, device=t.device)
        _copy_strided(shadow, t)
        shadow._spx_view = t
        t = shadow
    return _vec(t, like, name)


def _sync_shadow(t: Optional[torch.Tensor]) -> None:
    view = getattr(t, "_spx_view", None)
    if view is not None:
        _copy_strided(t, view)


def _p(t: Optional[torch.Tensor]) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


def _bound(b, like: torch.Tensor, name: str) -> L.Bound:
    if isinstance(b, torch.Tensor) and b.dim() > 0:
        _vec(b, like, name)
        return L.Bound(b.data_ptr(), 0.0)
    return L.Bound(None, float(b))


# ---------------------------------------------------------- base functions h ---
class NormL1:
    """ProximalOperators.NormL1(λ): λ‖x‖₁."""

    def __init__(self, lam: float = 1.0):
        if lam < 0:
            raise ValueError("parameter λ must be nonnegative")
        self.lam = float(lam)

    lambda_ = property(lambda self: self.lam)


class NormL0(NormL1):
    """ProximalOperators.NormL0(λ): λ·count(x ≠ 0)."""


class RootNormLhalf(NormL1):
    """RootNormLhalf(λ): λ Σ√|x_i|  (src/rootNormLhalf.jl:10-29)."""

    def __init__(self, lam: float = 1.0):
        if lam < 0:
            raise ValueError("λ must be nonnegative")  # rootNormLhalf.jl:17-18
        self.lam = float(lam)


class NormL2(NormL1):
    """ProximalOperators.NormL2(λ): λ‖x‖₂ (as h: one-group GroupNormL2; as χ: ℓ2 trust region)."""


class NormLinf(NormL1):
    """ProximalOperators.NormLinf(λ) = Conjugate(IndBallL1(λ)): the χ of the BInf trust regions."""


class IndBallL0:
    """ProximalOperators.IndBallL0(r): indicator of {‖x‖₀ ≤ r}."""

    def __init__(self, r: int):
        if r <= 0:
            raise ValueError("parameter r must be a positive integer")
        self.r = int(r)


class GroupNormL2:
    """GroupNormL2(λ, idx): Σ_g λ_g‖x[idx_g]‖₂  (src/groupNormL2.jl:15-39).

    `lambdas`: one weight per group; `idx`: list of Python ranges / (start, stop) pairs
    (0-based, stop exclusive) that partition 0..n-1 in order, or None for the single group
    `[:]` (groupNormL2.jl:30-31).  Device-side the layout is CSR offsets.
    """

    def __init__(self, lambdas: Sequence[float] = (1.0,), idx=None, offsets: Optional[torch.Tensor] = None):
        self.lambdas = lambdas
        if idx is not None and offsets is None:
            if not isinstance(lambdas, torch.Tensor) and len(lambdas) != len(idx):
                raise ValueError("number of weights and groups should be the same")  # groupNormL2.jl:20-23
            offs = [0]
            for g in idx:
                a, b = (g.start, g.stop) if isinstance(g, range) else (int(g[0]), int(g[1]))
                if a != offs[-1] or b < a:
                    raise ValueError("groups must be contiguous ranges that partition the vector in order")
                offs.append(b)
            self.offsets_host = offs
        else:
            self.offsets_host = None
        self.offsets = offsets
        self.idx = idx


# ------------------------------------------------------------ shifted types ---
class ShiftedProximableFunction:
    """abstract type ShiftedProximableFunction  (ShiftedProximalOperators.jl:18)."""

    h = None
    xk: torch.Tensor
    sj: torch.Tensor
    sol: torch.Tensor
    shifted_twice: bool

    def _init_common(self, h, xk, sj, shifted_twice):
        self.h = h
        self.xk = _adopt(xk, name="xk")  # aliased, not copied (shiftedNormL1.jl:16-25)
        self.sj = torch.zeros_like(self.xk) if sj is None else _adopt(sj, self.xk, "sj")
        self.sol = torch.empty_like(self.xk)
        self.shifted_twice = bool(shifted_twice)
        self._suf = _SUF[self.xk.dtype]

    # getproperty sugar: ψ.λ, ψ.r  (ShiftedProximalOperators.jl:113-121)
    @property
    def lam(self):
        return self.h.lam

    @property
    def r(self):
        return self.h.r

    @property
    def n(self):
        return self.xk.numel()

    def _ctx(self):
        return context(self.xk.device)

    def _call(self, name, *args):
        _sync_shadow(self.xk)  # strided SubArray shifts: refresh the contiguous shadows
        _sync_shadow(self.sj)
        L.call(f"spx_{name}_{self._suf}", self._ctx(), *args)

    def _check(self, y, q, names=("y", "q")):
        _vec(y, self.xk, names[0])
        _vec(q, self.xk, names[1])

    # generic ψ(y) = h(xk + sj + y)  (ShiftedProximalOperators.jl:51-54)
    _H_KIND = None

    def __call__(self, y: torch.Tensor) -> float:
        _vec(y, self.xk, "y")
        out = C.c_double()
        self._call("value_sep", C.c_int32(self._H_KIND), C.c_int64(self.n), _p(self.xk), _p(self.sj), _p(y),
                   C.c_double(getattr(self.h, "lam", 0.0)), C.c_int64(getattr(self.h, "r", 0)), C.byref(out))
        return out.value

    def prox_(self, y, q, sigma, want_value=False):
        raise NotImplementedError

    def iprox_(self, y, g, d, want_value=False):
        raise NotImplementedError(f"iprox! is not defined for {type(self).__name__}")

    def step_(self, s, grad, nu, xsy=None):
        """The solver step for the types whose prox! is not one streaming pass (groups, top-r, ShiftedNormL1B2): the
        caller's sweeps as two passes around the type's own prox! -- spx_step_pre_* writes q = -ν∇f where s will be,
        prox!(s, ψ, s, ν) runs in place with ψ(s) out of its own pass (or the type's ψ(y) entry), spx_step_post_* gives
        xsy = xk + sj + s, Σs² and Σ∇f·s in one pass.  Same results as the separate sweeps, bit for bit for s and xsy.
        The separable and Box types override this with the single-pass form."""
        self._check(s, grad, ("s", "grad"))
        if xsy is not None:
            _vec(xsy, self.xk, "xsy")
        if s.data_ptr() == grad.data_ptr():
            raise ValueError("step_: s must not alias grad")
        self._call("step_pre", C.c_int64(self.n), _p(s), _p(grad), C.c_double(nu))
        _, val = self.prox_(s, s, nu, want_value=True)
        out = (C.c_double * 2)()
        sj = self.sj if self.shifted_twice else None
        self._call("step_post", C.c_int64(self.n), _p(xsy), _p(self.xk), _p(sj), _p(s), _p(grad), out)
        return s, StepResult(val, math.sqrt(out[0]), out[1])

    def _step_sep(self, s, grad, nu, xsy):
        # spx_step_sep_*: q = -ν∇f, prox!, ψ(s), xk+sj+s, Σs², Σ∇f·s in the one pass of the prox!
        self._check(s, grad, ("s", "grad"))
        if xsy is not None:
            _vec(xsy, self.xk, "xsy")
        out = (C.c_double * 3)()
        # ψ shifted once: sj is the zero vector the constructor made (shift! then writes xk,
        # ShiftedProximalOperators.jl:72-79) -- NULL reads it as zeros without the traffic
        sj = self.sj if self.shifted_twice else None
        self._call("step_sep", C.c_int32(self._H_KIND), C.c_int64(self.n), _p(s), _p(xsy), _p(self.xk), _p(sj),
                   _p(grad), C.c_double(self.h.lam), C.c_double(nu), out)
        return s, StepResult(out[0], math.sqrt(out[1]), out[2])

    def istep_(self, s, grad, d, dshift=0.0, xsy=None):
        raise NotImplementedError(f"iprox! is not defined for {type(self).__name__}")

    def _istep_check(self, s, grad, d, xsy):
        self._check(s, grad, ("s", "grad"))
        _vec(d, self.xk, "d")
        if xsy is not None:
            _vec(xsy, self.xk, "xsy")

    def _istep_sep(self, s, grad, d, dshift, xsy):
        # spx_istep_sep_*: D + σ, iprox!, ψ(s), xk+sj+s, Σs², Σ∇f·s, Σ d s² in the one pass of the iprox!
        self._istep_check(s, grad, d, xsy)
        out = (C.c_double * 4)()
        bad = C.c_int64()
        sj = self.sj if self.shifted_twice else None  # ψ shifted once: NULL reads zeros (see _step_sep)
        self._call("istep_sep", C.c_int32(self._H_KIND), C.c_int64(self.n), _p(s), _p(xsy), _p(self.xk), _p(sj),
                   _p(grad), _p(d), C.c_double(dshift), C.c_double(self.h.lam), C.byref(bad), out)
        return s, IStepResult(out[0], math.sqrt(out[1]), out[2], out[3])

    def __repr__(self):  # Base.show  (ShiftedProximalOperators.jl:123-133)
        return f"{type(self).__name__}(n={self.n}, dtype={self.xk.dtype}, shifted_twice={self.shifted_twice})"


class StepResult(tuple):
    """(ψ(s), ‖s‖₂, ∇f·s) of a fused solver step."""
    __slots__ = ()

    def __new__(cls, psi, snorm, gdots):
        return super().__new__(cls, (psi, snorm, gdots))

    psi = property(lambda self: self[0])
    snorm = property(lambda self: self[1])
    gdots = property(lambda self: self[2])


class IStepResult(tuple):
    """(ψ(s), ‖s‖₂, ∇f·s, sᵀ(D + σ)s) of a fused solver step around iprox!."""
    __slots__ = ()

    def __new__(cls, psi, snorm, gdots, sds):
        return super().__new__(cls, (psi, snorm, gdots, sds))

    psi = property(lambda self: self[0])
    snorm = property(lambda self: self[1])
    gdots = property(lambda self: self[2])
    sds = property(lambda self: self[3])


def _psi_arg(want_value):
    out = C.c_double() if want_value else None
    return out, (C.byref(out) if want_value else None)


class ShiftedNormL1(ShiftedProximableFunction):
    """ShiftedNormL1  (src/shiftedNormL1.jl:3-34)."""
    _H_KIND = L.H_L1

    def __init__(self, h, xk, sj=None, shifted_twice=False):
        self._init_common(h, xk, sj, shifted_twice)

    def step_(self, s, grad, nu, xsy=None):
        return self._step_sep(s, grad, nu, xsy)

    def istep_(self, s, grad, d, dshift=0.0, xsy=None):
        return self._istep_sep(s, grad, d, dshift, xsy)

    def prox_(self, y, q, sigma, want_value=False):  # shiftedNormL1.jl:40-54
        self._check(y, q)
        out, ref = _psi_arg(want_value)
        self._call("prox_l1", C.c_int64(self.n), _p(y), _p(self.xk), _p(self.sj), _p(q), C.c_double(self.h.lam),
                   C.c_double(sigma), ref)
        return (y, out.value) if want_value else y

    def iprox_(self, y, g, d, want_value=False):  # shiftedNormL1.jl:60-75
        self._check(y, g, ("y", "g"))
        _vec(d, self.xk, "d")
        bad = C.c_int64()
        out, ref = _psi_arg(want_value)
        self._call("iprox_l1", C.c_int64(self.n), _p(y), _p(self.xk), _p(self.sj), _p(g), _p(d),
                   C.c_double(self.h.lam), C.byref(bad), ref)
        return (y, out.value) if want_value else y


class ShiftedNormL0(ShiftedProximableFunction):
    """ShiftedNormL0  (src/shiftedNormL0.jl:3-36)."""
    _H_KIND = L.H_L0

    def __init__(self, h, xk, sj=None, shifted_twice=False):
        self._init_common(h, xk, sj, shifted_twice)

    def step_(self, s, grad, nu, xsy=None):
        return self._step_sep(s, grad, nu, xsy)

    def istep_(self, s, grad, d, dshift=0.0, xsy=None):
        return self._istep_sep(s, grad, d, dshift, xsy)

    def prox_(self, y, q, sigma, want_value=False):  # shiftedNormL0.jl:38-55
        self._check(y, q)
        out, ref = _psi_arg(want_value)
        self._call("prox_l0", C.c_int64(self.n), _p(y), _p(self.xk), _p(self.sj), _p(q), C.c_double(self.h.lam),
                   C.c_double(sigma), ref)
        return (y, out.value) if want_value else y

    def iprox_(self, y, g, d, want_value=False):  # shiftedNormL0.jl:61-80
        self._check(y, g, ("y", "g"))
        _vec(d, self.xk, "d")
        bad = C.c_int64()
        out, ref = _psi_arg(want_value)
        self._call("iprox_l0", C.c_int64(self.n), _p(y), _p(self.xk), _p(self.sj), _p(g), _p(d),
                   C.c_double(self.h.lam), C.byref(bad), ref)
        return (y, out.value) if want_value else y


class ShiftedRootNormLhalf(ShiftedProximableFunction):
    """ShiftedRootNormLhalf  (src/shiftedRootNormLhalf.jl:4-35)."""
    _H_KIND = L.H_LHALF

    def __init__(self, h, xk, sj=None, shifted_twice=False):
        self._init_common(h, xk, sj, shifted_twice)

    def step_(self, s, grad, nu, xsy=None):
        return self._step_sep(s, grad, nu, xsy)

    def prox_(self, y, q, sigma, want_value=False):  # shiftedRootNormLhalf.jl:41-63
        self._check(y, q)
        out, ref = _psi_arg(want_value)
        self._call("prox_lhalf", C.c_int64(self.n), _p(y), _p(self.xk), _p(self.sj), _p(q), C.c_double(self.h.lam),
                   C.c_double(sigma), ref)
        return (y, out.value) if want_value else y


class _Selected:
    """`selected::AbstractArray{<:Integer}` on the device (spx_sel)."""

    def __init__(self, selected, n: int, device, ctx_fn):
        self.user = selected
        self.keep = []
        s = L.Sel(L.SEL_ALL, 0, 1, n - 1, None, None, 0)
        if selected is None:
            pass
        elif isinstance(selected, range):
            if selected.step <= 0:
                raise ValueError("selected: range step must be positive")
            if len(selected) == 0:
                s = L.Sel(L.SEL_RANGE, n, 1, n - 1, None, None, 0)
            else:
                s = L.Sel(L.SEL_RANGE, selected[0], selected.step, selected[-1], None, None, 0)
        else:
            lst = torch.as_tensor(selected, dtype=torch.int64).to(device).contiguous()
            mask = torch.empty((n + 31) // 32, dtype=torch.int32, device=device)
            L.call("spx_build_mask", ctx_fn(), C.c_int64(n), C.c_void_p(lst.data_ptr()), C.c_int64(lst.numel()),
                   C.c_void_p(mask.data_ptr()))
            self.keep = [lst, mask]
            s = L.Sel(L.SEL_MASK, 0, 1, n - 1, mask.data_ptr(), lst.data_ptr(), lst.numel())
        self.sel = s

    def ref(self):
        return C.byref(self.sel)


class _BoxBase(ShiftedProximableFunction):
    """Common part of ShiftedNormL1Box / ShiftedNormL0Box / ShiftedRootNormLhalfBox
    (src/shiftedNormL1Box.jl:3-68 and the two siblings)."""
    _BOX_NAME = ""
    _CHECK_BOUNDS = True

    def __init__(self, h, xk, sj, l, u, shifted_twice=False, selected=None):
        self._init_common(h, xk, sj, shifted_twice)
        self.l, self.u = l, u
        self._sel = selected if isinstance(selected, _Selected) else _Selected(selected, self.n, xk.device, self._ctx)
        self.selected = self._sel.user if self._sel.user is not None else range(self.n)
        if self._CHECK_BOUNDS:  # `any(l .> u)` -> error  (shiftedNormL1Box.jl:33-35, shiftedNormL0Box.jl:33-35)
            flag = C.c_int32()
            lb, ub = _bound(l, xk, "l"), _bound(u, xk, "u")
            self._call("any_gt", C.c_int64(self.n), C.byref(lb), C.byref(ub), C.byref(flag))
            if flag.value:
                raise ValueError("Error: at least one lower bound is greater than the upper bound.")

    def _bounds(self):
        return _bound(self.l, self.xk, "l"), _bound(self.u, self.xk, "u")

    def prox_(self, y, q, sigma, want_value=False):
        self._check(y, q)
        lb, ub = self._bounds()
        out, ref = _psi_arg(want_value)
        self._call(f"prox_{self._BOX_NAME}", C.c_int64(self.n), _p(y), _p(self.xk), _p(self.sj), _p(q), C.byref(lb),
                   C.byref(ub), self._sel.ref(), C.c_double(self.h.lam), C.c_double(sigma), ref)
        return (y, out.value) if want_value else y

    def iprox_(self, y, g, d, want_value=False):
        if self._BOX_NAME == "lhalfbox":
            raise NotImplementedError("iprox! is not defined for ShiftedRootNormLhalfBox")
        self._check(y, g, ("y", "g"))
        _vec(d, self.xk, "d")
        lb, ub = self._bounds()
        out, ref = _psi_arg(want_value)
        self._call(f"iprox_{self._BOX_NAME}", C.c_int64(self.n), _p(y), _p(self.xk), _p(self.sj), _p(g), _p(d),
                   C.byref(lb), C.byref(ub), self._sel.ref(), C.c_double(self.h.lam), ref)
        return (y, out.value) if want_value else y

    def step_(self, s, grad, nu, xsy=None):
        self._check(s, grad, ("s", "grad"))
        if xsy is not None:
            _vec(xsy, self.xk, "xsy")
        lb, ub = self._bounds()
        out = (C.c_double * 3)()
        self._call("step_box", C.c_int32(_BOX_OP[self._BOX_NAME]), C.c_int64(self.n), _p(s), _p(xsy), _p(self.xk),
                   _p(self.sj), _p(grad), C.byref(lb), C.byref(ub), self._sel.ref(), C.c_double(self.h.lam),
                   C.c_double(nu), out)
        return s, StepResult(out[0], math.sqrt(out[1]), out[2])

    def istep_(self, s, grad, d, dshift=0.0, xsy=None):
        if self._BOX_NAME == "lhalfbox":
            raise NotImplementedError("iprox! is not defined for ShiftedRootNormLhalfBox")
        self._istep_check(s, grad, d, xsy)
        lb, ub = self._bounds()
        out = (C.c_double * 4)()
        self._call("istep_box", C.c_int32(_BOX_OP[self._BOX_NAME]), C.c_int64(self.n), _p(s), _p(xsy), _p(self.xk),
                   _p(self.sj), _p(grad), _p(d), C.c_double(dshift), C.byref(lb), C.byref(ub), self._sel.ref(),
                   C.c_double(self.h.lam), out)
        return s, IStepResult(out[0], math.sqrt(out[1]), out[2], out[3])

    def __call__(self, y):  # shiftedNormL1Box.jl:70-82
        _vec(y, self.xk, "y")
        lb, ub = self._bounds()
        out = C.c_double()
        self._call("value_box", C.c_int32(self._H_KIND), C.c_int64(self.n), _p(self.xk), _p(self.sj), _p(y),
                   C.byref(lb), C.byref(ub), self._sel.ref(), C.c_double(self.h.lam), C.byref(out))
        return out.value


class ShiftedNormL1Box(_BoxBase):
    """prox! shiftedNormL1Box.jl:89-125, iprox! :131-225."""
    _H_KIND, _BOX_NAME = L.H_L1, "l1box"


class ShiftedNormL0Box(_BoxBase):
    """prox! shiftedNormL0Box.jl:89-131, iprox! :137-231."""
    _H_KIND, _BOX_NAME = L.H_L0, "l0box"


class ShiftedRootNormLhalfBox(_BoxBase):
    """prox! shiftedRootNormLhalfBox.jl:86-120 (its constructor has no l > u check, :20-45)."""
    _H_KIND, _BOX_NAME, _CHECK_BOUNDS = L.H_LHALF, "lhalfbox", False


class ShiftedNormL1B2(ShiftedProximableFunction):
    """ShiftedNormL1B2  (src/shiftedNormL1B2.jl:3-40)."""
    _H_KIND = L.H_L1

    def __init__(self, h, xk, sj, Delta, chi, shifted_twice=False):
        self._init_common(h, xk, sj, shifted_twice)
        self.Delta, self.chi = float(Delta), chi
        self.last_passes = 0

    def prox_(self, y, q, sigma, want_value=False):  # shiftedNormL1B2.jl:47-64
        self._check(y, q)
        passes = C.c_int32()
        out, ref = _psi_arg(want_value)
        self._call("prox_l1b2", C.c_int64(self.n), _p(y), _p(self.xk), _p(self.sj), _p(q), C.c_double(self.h.lam),
                   C.c_double(sigma), C.c_double(self.Delta), C.c_double(self.chi.lam), C.byref(passes), ref)
        self.last_passes = passes.value
        return (y, out.value) if want_value else y

    def _step_args(self, s, grad, nu, xsy):
        self._check(s, grad, ("s", "grad"))
        if xsy is not None:
            _vec(xsy, self.xk, "xsy")
        span = s.numel() * s.element_size()
        if s.numel() > 0 and abs(s.data_ptr() - grad.data_ptr()) < span:
            raise ValueError("step_: s must not overlap grad")
        if s.numel() > 0 and xsy is not None and abs(s.data_ptr() - xsy.data_ptr()) < span:
            raise ValueError("step_: xsy must not overlap s")
        return (C.c_int64(self.n), _p(s), _p(xsy), _p(self.xk), _p(self.sj), _p(grad), C.c_double(self.h.lam),
                C.c_double(nu), C.c_double(self.Delta), C.c_double(self.chi.lam))

    def step_(self, s, grad, nu, xsy=None):
        """spx_step_l1b2_*: the whole step inside the passes of prox!'s own root search -- q = -ν∇f is formed from ∇f
        in every pass, the finish writes s and xsy and sums ψ(s), Σs², Σ∇f·s.  s is bit-identical to
        prox_(y, ψ, -ν∇f, ν) into a y that overlaps no input; `last_passes` is set as by prox_."""
        out, passes = (C.c_double * 3)(), C.c_int32()
        self._call("step_l1b2", *self._step_args(s, grad, nu, xsy), C.byref(passes), out)
        self.last_passes = passes.value
        return s, StepResult(out[0], math.sqrt(out[1]), out[2])

    def __call__(self, y):  # shiftedNormL1B2.jl:32
        _vec(y, self.xk, "y")
        out = C.c_double()
        self._call("value_l1b2", C.c_int64(self.n), _p(self.xk), _p(self.sj), _p(y), C.c_double(self.h.lam),
                   C.c_double(self.Delta), C.byref(out))
        return out.value


def _step_indballl0(psi, s, grad, nu, xsy, binf, delta):
    # spx_step_indballl0_*: the whole step in one pass of the stream top-r kernel on a batch it takes, the composed form
    # (step_pre, prox! in place, ψ(s), step_post) otherwise -- decided in the library
    psi._check(s, grad, ("s", "grad"))
    if xsy is not None:
        _vec(xsy, psi.xk, "xsy")
    if s.numel() > 0 and s.data_ptr() == grad.data_ptr():
        raise ValueError("step_: s must not alias grad")
    out = (C.c_double * 3)()
    psi._call("step_indballl0", C.c_int64(psi.nprob), C.c_int64(psi.n // psi.nprob), _p(s), _p(xsy), _p(psi.xk),
              _p(psi.sj), _p(grad), C.c_int64(psi.h.r), C.c_int32(binf), C.c_double(delta), C.c_double(nu), out)
    return s, StepResult(out[0], math.sqrt(out[1]), out[2])


class ShiftedIndBallL0(ShiftedProximableFunction):
    """ShiftedIndBallL0  (src/shiftedIndBallL0.jl:3-49); the `p` permutation scratch does not exist here."""
    _H_KIND = L.H_INDBALLL0

    def __init__(self, h, xk, sj=None, shifted_twice=False, nprob: int = 1):
        self._init_common(h, xk, sj, shifted_twice)
        if self.n % nprob:
            raise ValueError("vector length must be a multiple of the number of problems")
        self.nprob = int(nprob)

    def prox_(self, y, q, sigma=None, want_value=False):  # shiftedIndBallL0.jl:54-72
        self._check(y, q)
        self._call("prox_indballl0", C.c_int64(self.nprob), C.c_int64(self.n // self.nprob), _p(y), _p(self.xk),
                   _p(self.sj), _p(q), C.c_int64(self.h.r), C.c_int32(0), C.c_double(0.0))
        return (y, self(y)) if want_value else y

    def step_(self, s, grad, nu, xsy=None):
        """spx_step_indballl0_*: the whole step in one pass of the stream top-r kernel for a batch of >= 2 problems per
        SM (the C5 shape), the two passes around prox! otherwise."""
        return _step_indballl0(self, s, grad, nu, xsy, 0, 0.0)


class ShiftedIndBallL0BInf(ShiftedProximableFunction):
    """ShiftedIndBallL0BInf  (src/shiftedIndBallL0BInf.jl:3-66)."""
    _H_KIND = L.H_INDBALLL0

    def __init__(self, h, xk, sj, Delta, chi, shifted_twice=False, nprob: int = 1):
        self._init_common(h, xk, sj, shifted_twice)
        self.Delta, self.chi = float(Delta), chi
        if self.n % nprob:
            raise ValueError("vector length must be a multiple of the number of problems")
        self.nprob = int(nprob)

    def prox_(self, y, q, sigma=None, want_value=False):  # shiftedIndBallL0BInf.jl:73-95
        self._check(y, q)
        self._call("prox_indballl0", C.c_int64(self.nprob), C.c_int64(self.n // self.nprob), _p(y), _p(self.xk),
                   _p(self.sj), _p(q), C.c_int64(self.h.r), C.c_int32(1), C.c_double(self.Delta))
        return (y, self(y)) if want_value else y

    def step_(self, s, grad, nu, xsy=None):
        """spx_step_indballl0_*: as ShiftedIndBallL0.step_, with ψ(s) = Inf when sj + s leaves the ball of 1.1Δ."""
        return _step_indballl0(self, s, grad, nu, xsy, 1, self.Delta)

    def __call__(self, y):  # shiftedIndBallL0BInf.jl:44-49
        _vec(y, self.xk, "y")
        out = C.c_double()
        self._call("value_binf", C.c_int32(L.H_INDBALLL0), C.c_int64(self.n), _p(self.xk), _p(self.sj), _p(y),
                   C.c_double(self.Delta), C.c_int64(self.h.r), C.c_int64(0), None, None, C.byref(out))
        return out.value


class _GroupBase(ShiftedProximableFunction):
    def _init_groups(self, h, xk):
        dt, dev = xk.dtype, xk.device
        if isinstance(h, NormL2):  # shifted(h::NormL2, xk) -> one group [:]  (shiftedGroupNormL2.jl:34-35)
            h = GroupNormL2([h.lam], None)
        if h.offsets is not None:
            self._offs = h.offsets.to(device=dev, dtype=torch.int64).contiguous()
        else:
            offs = h.offsets_host if h.offsets_host is not None else [0, xk.numel()]
            self._offs = torch.tensor(offs, dtype=torch.int64, device=dev)
        lam = h.lambdas
        self._lam_g = (lam.to(device=dev, dtype=dt) if isinstance(lam, torch.Tensor)
                       else torch.tensor(list(lam), dtype=dt, device=dev)).contiguous()
        self.ngroups = self._offs.numel() - 1
        if self._lam_g.numel() != self.ngroups:
            raise ValueError("number of weights and groups should be the same")
        # the device layout is checked once here and trusted by the kernels afterwards; the same pass records which
        # group-size classes the layout holds, so the entry points launch only the kernels that have work
        try:
            L.call("spx_group_validate_offsets", context(dev), C.c_int64(xk.numel()), C.c_int64(self.ngroups),
                   _p(self._offs))
        except SpxError as e:
            raise ValueError(str(e)) from None
        return h

    @property
    def lam(self):
        return self._lam_g


class ShiftedGroupNormL2(_GroupBase):
    """ShiftedGroupNormL2  (src/shiftedGroupNormL2.jl:3-46)."""

    def __init__(self, h, xk, sj=None, shifted_twice=False):
        self._init_common(h, xk, sj, shifted_twice)
        self.h = self._init_groups(h, xk)

    def prox_(self, y, q, sigma, want_value=False):  # shiftedGroupNormL2.jl:52-79
        self._check(y, q)
        out, ref = _psi_arg(want_value)
        self._call("prox_groupl2", C.c_int64(self.n), _p(y), _p(self.xk), _p(self.sj), _p(q), C.c_int64(self.ngroups),
                   _p(self._offs), _p(self._lam_g), C.c_double(sigma), ref)
        return (y, out.value) if want_value else y

    def __call__(self, y):  # ShiftedProximalOperators.jl:51-54 + groupNormL2.jl:33-39
        _vec(y, self.xk, "y")
        out = C.c_double()
        self._call("value_groupl2", C.c_int64(self.n), _p(self.xk), _p(self.sj), _p(y), C.c_int64(self.ngroups),
                   _p(self._offs), _p(self._lam_g), C.byref(out))
        return out.value

    def step_(self, s, grad, nu, xsy=None):
        """spx_step_groupl2_*: the whole step in one pass when every group holds <= 256 elements (the C4 shape), the
        two passes around prox! otherwise (decided in the library from the census of the validated layout)."""
        self._check(s, grad, ("s", "grad"))
        if xsy is not None:
            _vec(xsy, self.xk, "xsy")
        if s.data_ptr() == grad.data_ptr():
            raise ValueError("step_: s must not alias grad")
        out = (C.c_double * 3)()
        self._call("step_groupl2", C.c_int64(self.n), _p(s), _p(xsy), _p(self.xk), _p(self.sj), _p(grad),
                   C.c_int64(self.ngroups), _p(self._offs), _p(self._lam_g), C.c_double(nu), out)
        return s, StepResult(out[0], math.sqrt(out[1]), out[2])


class ShiftedGroupNormL2Binf(_GroupBase):
    """ShiftedGroupNormL2Binf  (src/shiftedGroupNormL2Binf.jl:3-60)."""

    def __init__(self, h, xk, sj, Delta, chi, shifted_twice=False):
        self._init_common(h, xk, sj, shifted_twice)
        self.h = self._init_groups(h, xk)
        self.Delta, self.chi = float(Delta), chi

    def prox_(self, y, q, sigma, want_value=False):  # shiftedGroupNormL2Binf.jl:67-119
        self._check(y, q)
        out, ref = _psi_arg(want_value)
        self._call("prox_groupl2binf", C.c_int64(self.n), _p(y), _p(self.xk), _p(self.sj), _p(q),
                   C.c_int64(self.ngroups), _p(self._offs), _p(self._lam_g), C.c_double(sigma),
                   C.c_double(self.Delta), ref)
        return (y, out.value) if want_value else y

    def __call__(self, y):  # shiftedGroupNormL2Binf.jl:34-39
        _vec(y, self.xk, "y")
        out = C.c_double()
        self._call("value_binf", C.c_int32(L.H_GROUPL2), C.c_int64(self.n), _p(self.xk), _p(self.sj), _p(y),
                   C.c_double(self.Delta), C.c_int64(0), C.c_int64(self.ngroups), _p(self._offs), _p(self._lam_g),
                   C.byref(out))
        return out.value

    def step_(self, s, grad, nu, xsy=None):
        """spx_step_groupl2binf_*: the whole step in one pass on a uniform layout (n == ngroups m, m = 16 ... 256, the
        C4 shape), the two passes around prox! otherwise (decided in the library)."""
        self._check(s, grad, ("s", "grad"))
        if xsy is not None:
            _vec(xsy, self.xk, "xsy")
        if s.numel() > 0 and s.data_ptr() == grad.data_ptr():
            raise ValueError("step_: s must not alias grad")
        out = (C.c_double * 3)()
        self._call("step_groupl2binf", C.c_int64(self.n), _p(s), _p(xsy), _p(self.xk), _p(self.sj), _p(grad),
                   C.c_int64(self.ngroups), _p(self._offs), _p(self._lam_g), C.c_double(nu), C.c_double(self.Delta),
                   out)
        return s, StepResult(out[0], math.sqrt(out[1]), out[2])


# ------------------------------------------------------------------- verbs ---
_PLAIN = {NormL1: ShiftedNormL1, NormL0: ShiftedNormL0, RootNormLhalf: ShiftedRootNormLhalf}
_BOX = {NormL1: ShiftedNormL1Box, NormL0: ShiftedNormL0Box, RootNormLhalf: ShiftedRootNormLhalfBox}


def shifted(h, x, *args, selected=None, nprob: int = 1):
    """`shifted(...)`: the constructor table of SURVEY.md §3.1.

    shifted(h, xk)                      shiftedNormL1.jl:28-29 and siblings
    shifted(h, xk, l, u[, selected])    shiftedNormL1Box.jl:50-56 and siblings
    shifted(h, xk, Δ, χ[, selected])    :57-63 (χ = NormLinf -> Box with ±Δ); NormL2 χ -> ShiftedNormL1B2
    shifted(ψ, sj)                      second shift, shares ψ.xk, shifted_twice = true
    `nprob` (extension): the IndBallL0 types can hold a batch of independent problems back to back.
    """
    if isinstance(h, ShiftedProximableFunction):  # shifted(ψ, sj)
        psi, sj = h, _adopt(x, h.xk, "sj")
        if isinstance(psi, _BoxBase):
            return type(psi)(psi.h, psi.xk, sj, psi.l, psi.u, True, psi._sel)
        if isinstance(psi, (ShiftedNormL1B2, ShiftedGroupNormL2Binf)):
            return type(psi)(psi.h, psi.xk, sj, psi.Delta, psi.chi, True)
        if isinstance(psi, ShiftedIndBallL0BInf):
            return ShiftedIndBallL0BInf(psi.h, psi.xk, sj, psi.Delta, psi.chi, True, psi.nprob)
        if isinstance(psi, ShiftedIndBallL0):
            return ShiftedIndBallL0(psi.h, psi.xk, sj, True, psi.nprob)
        return type(psi)(psi.h, psi.xk, sj, True)
    xk = _adopt(x, name="xk")
    if len(args) == 0:
        if type(h) in _PLAIN:
            return _PLAIN[type(h)](h, xk)
        if isinstance(h, (GroupNormL2, NormL2)):
            return ShiftedGroupNormL2(h, xk)
        if isinstance(h, IndBallL0):
            return ShiftedIndBallL0(h, xk, nprob=nprob)
        raise TypeError(f"shifted: unsupported h {type(h).__name__}")
    if len(args) == 3 and selected is None:
        args, selected = args[:2], args[2]
    if len(args) != 2:
        raise TypeError("shifted(h, x, l, u[, selected]) or shifted(h, x, Δ, χ[, selected])")
    a, b = args
    if isinstance(b, NormLinf):  # BInf trust region
        delta = float(a)
        if type(h) in _BOX:
            return _BOX[type(h)](h, xk, None, -delta, delta, False, selected)
        if isinstance(h, (GroupNormL2, NormL2)):
            return ShiftedGroupNormL2Binf(h, xk, None, delta, b)
        if isinstance(h, IndBallL0):
            return ShiftedIndBallL0BInf(h, xk, None, delta, b, nprob=nprob)
        raise TypeError(f"shifted: unsupported h {type(h).__name__} with an ℓ∞ trust region")
    if isinstance(b, NormL2):  # ℓ2 trust region
        if type(h) is NormL1:
            return ShiftedNormL1B2(h, xk, None, float(a), b)
        raise TypeError("shifted: the ℓ2 trust region is defined for NormL1 only (shiftedNormL1B2.jl:34-35)")
    if type(h) in _BOX:
        return _BOX[type(h)](h, xk, None, a, b, False, selected)
    raise TypeError(f"shifted: unsupported h {type(h).__name__} with bounds")


def shift_(psi, v):
    """shift!(ψ, v): ψ.sj .= v if shifted twice else ψ.xk .= v  (ShiftedProximalOperators.jl:72-79).
    Copies INTO the aliased array, like the reference."""
    dst = psi.sj if psi.shifted_twice else psi.xk
    _vec(v, dst, "shift")
    L.call("spx_memcpy_d2d", psi._ctx(), _p(dst), _p(v), C.c_size_t(dst.numel() * dst.element_size()))
    view = getattr(dst, "_spx_view", None)
    if view is not None:  # strided SubArray shift: write through into the caller's parent array
        _copy_strided(view, dst)
    return psi


def set_bounds_(psi, l, u):
    """set_bounds!(ψ, l, u)  (ShiftedProximalOperators.jl:107-111): vector bounds are copied into ψ.l / ψ.u."""
    if not isinstance(psi, _BoxBase):
        raise TypeError("set_bounds! is defined for the Box types only")
    for name, new in (("l", l), ("u", u)):
        cur = getattr(psi, name)
        if isinstance(cur, torch.Tensor) and cur.dim() > 0:
            if isinstance(new, torch.Tensor) and new.dim() > 0:
                _vec(new, cur, name)
                L.call("spx_memcpy_d2d", psi._ctx(), _p(cur), _p(new), C.c_size_t(cur.numel() * cur.element_size()))
            else:
                L.call(f"spx_fill_{psi._suf}", psi._ctx(), _p(cur), C.c_int64(cur.numel()), _CT[cur.dtype](float(new)))
        else:
            setattr(psi, name, new if isinstance(new, torch.Tensor) and new.dim() > 0 else float(new))
    return psi


def set_radius_(psi, delta):
    """set_radius!(ψ, Δ)  (ShiftedProximalOperators.jl:93-99): Box types -> set_bounds!(ψ, -Δ, Δ)."""
    if isinstance(psi, _BoxBase):
        return set_bounds_(psi, -float(delta), float(delta))
    if not hasattr(psi, "Delta"):
        raise TypeError(f"set_radius! is not defined for {type(psi).__name__}")
    psi.Delta = float(delta)
    return psi


def _prox_base_(y, h, x, gamma):
    """prox!(y, h, x, γ) of the in-tree base functions -- RootNormLhalf (src/rootNormLhalf.jl:31-51) and
    GroupNormL2 (src/groupNormL2.jl:41-58): same kernels as the shifted forms with the shifts read as zeros
    (NULL pointers: nothing extra crosses HBM).  Returns (y, value) with the reference's return value, out of
    the same pass: λ Σ√|y_i| for RootNormLhalf, Σ_g λ_g ‖x_g‖ -- the norms of the INPUT -- for GroupNormL2
    (groupNormL2.jl:49-54)."""
    _vec(x, name="x")
    _vec(y, x, "y")
    suf = _SUF[x.dtype]
    out = C.c_double()
    ctx = context(x.device)
    if isinstance(h, RootNormLhalf):
        L.call(f"spx_prox_lhalf_{suf}", ctx, C.c_int64(x.numel()), _p(y), None, None, _p(x), C.c_double(h.lam),
               C.c_double(gamma), C.byref(out))
    else:
        g = _GroupBase.__new__(_GroupBase)
        g._init_groups(h, x)
        L.call(f"spx_prox_groupl2_{suf}", ctx, C.c_int64(x.numel()), _p(y), None, None, _p(x), C.c_int64(g.ngroups),
               _p(g._offs), _p(g._lam_g), C.c_double(gamma), C.byref(out))
    return y, out.value


def prox_(y, psi, q, sigma, want_value=False):
    """prox!(y, ψ, q, σ).  `want_value=True` (extension) also returns ψ(y), fused into the same pass.
    With a base function (RootNormLhalf, GroupNormL2) instead of a shifted ψ: prox!(y, h, x, γ) -> (y, value)."""
    if isinstance(psi, (RootNormLhalf, GroupNormL2)):
        return _prox_base_(y, psi, q, sigma)
    return psi.prox_(y, q, sigma, want_value)


def prox(psi, q, sigma):
    """prox(ψ, q, σ) = prox!(ψ.sol, ψ, q, σ)  (ShiftedProximalOperators.jl:189-190)."""
    return psi.prox_(psi.sol, q, sigma)


def iprox_(y, psi, g, d, want_value=False):
    """iprox!(y, ψ, g, d)."""
    return psi.iprox_(y, g, d, want_value)


def iprox(psi, g, d):
    """iprox(ψ, g, d) = iprox!(ψ.sol, ψ, g, d)  (ShiftedProximalOperators.jl:180)."""
    return psi.iprox_(psi.sol, g, d)


def step_(s, psi, grad, nu, xsy=None):
    """Fused solver step (extension, SURVEY.md §8f rank 1): what an R2 / TR iteration of the reference's callers
    (README.md:17) wraps around its prox!, in the one pass of the prox! itself --

        q = -ν .* ∇f;  prox!(s, ψ, q, ν);  xsy .= xk .+ sj .+ s (if given);  ψ(s);  ‖s‖₂;  ∇f's

    Returns (s, StepResult(psi, snorm, gdots)).  `s` is bit-identical to prox_(s, ψ, -ν*grad, ν).  One pass for
    ShiftedNormL1 / L0 / RootNormLhalf and their Box / BInf forms; for the group, top-r and L1B2 types the sweeps are
    two passes around the type's own prox! (ShiftedProximableFunction.step_)."""
    return psi.step_(s, grad, nu, xsy)


def istep_(s, psi, grad, d, dshift=0.0, xsy=None):
    """Fused solver step around iprox! (extension): what an iteration of a diagonal quasi-Newton solver (R2DH, TRDH
    of RegularizedOptimization.jl) wraps around its iprox!, in the one pass of the iprox! itself --

        d = D .+ σ;  iprox!(s, ψ, ∇f, d);  xsy .= xk .+ sj .+ s (if given);  ψ(s);  ‖s‖₂;  ∇f's;  sᵀ d s

    with D = `d` and σ = `dshift`.  Returns (s, IStepResult(psi, snorm, gdots, sds)).  `s` is bit-identical to
    iprox_(s, ψ, grad, D + σ) with D + σ rounded to the vector's type; the sums are in Float64.  ShiftedNormL1 /
    ShiftedNormL0 raise AssertionError on a d[i] <= 0, as their iprox! does.  Defined for the types with an iprox!:
    ShiftedNormL1, ShiftedNormL0, ShiftedNormL1Box, ShiftedNormL0Box.  `s` may be `grad` and `xsy` may be ψ.xk."""
    return psi.istep_(s, grad, d, dshift, xsy)


def prox_zero(q, l, u):
    """prox_zero  (ShiftedProximalOperators.jl:203)."""
    f = L.lib().spx_prox_zero_f64
    f.restype = C.c_double
    return f(C.c_double(q), C.c_double(l), C.c_double(u))


def iprox_zero(d, g, l, u):
    """iprox_zero  (ShiftedProximalOperators.jl:217-236)."""
    f = L.lib().spx_iprox_zero_f64
    f.restype = C.c_double
    return f(C.c_double(d), C.c_double(g), C.c_double(l), C.c_double(u))
