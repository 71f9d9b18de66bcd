"""Host-side mirror of the LinearMixingModels.jl / AbstractGPs interface for the inference hot
path, on top of the liblmm C ABI (include/lmm.h).

Julia is not installed in the build image, so this Python layer plays the role of the Julia shim
(`julia/LinearMixingModelsB200.jl` holds the ccall version a maintainer would load): same
exported names (src/LinearMixingModels.jl:21-24), same argument meaning, same error behaviour:

    f  = ILMM(independent_mogp([GP(SEKernel()), GP(Matern32Kernel())]), Orthogonal(U, S))
    fx = f(MOInputIsotopicByOutputs(x, p), 0.1)
    logpdf(fx, y); post = posterior(fx, y); mean_and_var(post(x_test, 0.1)); rand(rng, fx)

Dispatch mirrors the reference: `H` an `Orthogonal` => OILMM path (src/oilmm.jl:13), a plain
matrix => general ILMM (src/ilmm.jl); inputs must be `MOInputIsotopicByOutputs` with scalar noise
(src/ilmm.jl:45) -- anything else raises TypeError (Julia: MethodError).  All numerics run in
liblmm on the GPU; nothing here computes on the CPU beyond argument marshalling.
"""
from __future__ import annotations

import ctypes as C
import os
import math
import weakref
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple, Union

import numpy as np

from . import _lib
from ._lib import GpDesc, PosDefException, as_f64, ptr

__all__ = [
    "SEKernel", "SqExponentialKernel", "Matern32Kernel", "Matern52Kernel", "ExponentialKernel", "Matern12Kernel", "RationalQuadraticKernel", "PeriodicKernel", "ScaleTransform", "ARDTransform", "with_lengthscale",
    "GP", "MOInputIsotopicByOutputs", "MOInputIsotopicByFeatures", "ColVecs", "RowVecs",
    "ILMM", "OILMM", "Orthogonal", "IndependentMOGP", "independent_mogp", "get_latent_gp",
    "FiniteGP", "Normal", "logpdf", "posterior", "mean_and_var", "mean", "var", "marginals", "rand", "cov", "mean_and_cov",
    "PosDefException", "Context", "default_context", "noise_var", "reshape_y", "unpack",
    "indices_which_reorder_outputs_to_features", "indices_which_reorder_features_to_outputs",
]


# --------------------------------------------------------------------------------------------
# context
# --------------------------------------------------------------------------------------------
class Context:
    """Owns one `lmm_ctx` (device, stream, memory pool, optional NCCL communicator)."""

    def __init__(self, device: Optional[int] = None):
        self.lib = _lib.load()
        if device is None:
            device = _current_device()
        h = C.c_void_p()
        rc = self.lib.lmm_ctx_create(int(device), C.byref(h))
        if rc != 0:
            raise RuntimeError(
                f"lmm_ctx_create(device={device}) failed with code {rc}: a CUDA device is required "
                "(liblmm has no CPU fallback)"
            )
        self.handle = h
        self.device = int(device)
        self.nranks, self.rank = 1, 0
        self._finalizer = weakref.finalize(self, self.lib.lmm_ctx_destroy, h)

    # -- helpers
    def error(self) -> str:
        return (self.lib.lmm_last_error(self.handle) or b"").decode()

    def set_option(self, key: str, value: float) -> None:
        rc = self.lib.lmm_ctx_set_option(self.handle, key.encode(), float(value))
        if rc != 0:
            raise ValueError(self.error())

    def counters(self) -> Tuple[int, int, int]:
        a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
        self.lib.lmm_ctx_counters(self.handle, C.byref(a), C.byref(b), C.byref(c))
        return a.value, b.value, c.value

    def last_timings(self) -> np.ndarray:
        out = np.zeros(8)
        self.lib.lmm_ctx_last_timings(self.handle, out.ctypes.data_as(C.POINTER(C.c_double)))
        return out

    def set_shard(self, nranks: int, rank: int) -> None:
        rc = self.lib.lmm_comm_set_shard(self.handle, nranks, rank)
        if rc != 0:
            raise ValueError("bad shard")
        self.nranks, self.rank = nranks, rank

    def init_nccl(self, unique_id: bytes, nranks: int, rank: int) -> None:
        buf = C.create_string_buffer(unique_id, 128)
        rc = self.lib.lmm_comm_init(self.handle, C.cast(buf, C.c_void_p), nranks, rank)
        if rc != 0:
            raise RuntimeError(f"lmm_comm_init failed ({rc}): {self.error()}")
        self.nranks, self.rank = nranks, rank

    def check(self, rc: int, info_latent: int = -1):
        if rc == 0:
            return
        msg = self.error()
        if rc > 0:
            raise PosDefException(rc, info_latent, msg)
        if rc == _lib.LMM_E_OUT_DIM:
            raise RuntimeError("out dim of x != out dim of f.")  # src/ilmm.jl:52
        if rc == _lib.LMM_E_NOT_ORTHOGONAL:
            raise ValueError("`U` is not an orthogonal matrix")
        if rc == _lib.LMM_E_OOM:
            raise MemoryError(msg)
        if rc in (_lib.LMM_E_ARG, _lib.LMM_E_UNSUPPORTED):
            raise ValueError(msg)
        raise RuntimeError(f"liblmm error {rc}: {msg}")


def _current_device() -> int:
    try:
        import torch

        if torch.cuda.is_available():
            return torch.cuda.current_device()
    except Exception:
        pass
    return 0


_default_ctx: Optional[Context] = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context()
    return _default_ctx


def set_default_context(ctx: Optional[Context]) -> None:
    global _default_ctx
    _default_ctx = ctx


# --------------------------------------------------------------------------------------------
# kernels, GP, inputs (KernelFunctions / AbstractGPs names)
# --------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Kernel:
    """`variance * (base ∘ ScaleTransform(inv_lengthscale) [∘ ARDTransform(ard)])`, optionally a flat KernelSum / KernelProduct
    (`k1 + k2`, `k1 * k2`, up to 4 terms) of such kernels: `terms` holds the further terms, `op` 1 = sum, 2 = product."""

    kind: int
    variance: float = 1.0
    inv_lengthscale: float = 1.0
    ard: Optional[tuple] = None  # ARDTransform multipliers (one per input dimension)
    param: float = 1.0  # shape parameter of the base kernel (α of RationalQuadraticKernel, r of PeriodicKernel)
    op: int = 0  # 0 single kernel, 1 KernelSum, 2 KernelProduct (LMM_COMPOSE_*)
    terms: tuple = ()  # the further terms of a composite kernel (single Kernels)

    def _single(self) -> "Kernel":
        return Kernel(self.kind, self.variance, self.inv_lengthscale, self.ard, self.param)

    def all_terms(self) -> tuple:
        return (self._single(),) + self.terms

    @property
    def kdiag(self) -> float:
        """k(x, x): κ(0) = 1 for every supported base kernel, so the sum / product of the term variances."""
        v = self.variance
        for t in self.terms:
            v = v * t.variance if self.op == 2 else v + t.variance
        return v

    @staticmethod
    def _from_terms(op: int, ts: tuple) -> "Kernel":
        if len(ts) > 4:
            raise TypeError("a composite kernel has at most 4 terms (LMM_MAX_TERMS)")
        t0 = ts[0]
        return Kernel(t0.kind, t0.variance, t0.inv_lengthscale, t0.ard, t0.param, op if len(ts) > 1 else 0, tuple(ts[1:]))

    @staticmethod
    def _combine(op: int, a: "Kernel", b: "Kernel") -> "Kernel":
        for k in (a, b):
            if k.op not in (0, op):
                raise TypeError("liblmm supports flat sums or flat products of base kernels (no sum of products / product of sums)")
        return Kernel._from_terms(op, a.all_terms() + b.all_terms())

    def __add__(self, other):  # KernelFunctions `k1 + k2` -> KernelSum
        if not isinstance(other, Kernel):
            return NotImplemented
        return Kernel._combine(1, self, other)

    def __rmul__(self, s):  # `0.5 * SEKernel()` -> ScaledKernel
        if not (isinstance(s, (int, float)) and s > 0):
            raise TypeError("kernel scale must be a positive real")
        if self.op == 1:  # c (k1 + k2) = c k1 + c k2
            return Kernel._from_terms(1, tuple(Kernel(t.kind, t.variance * float(s), t.inv_lengthscale, t.ard, t.param) for t in self.all_terms()))
        return Kernel(self.kind, self.variance * float(s), self.inv_lengthscale, self.ard, self.param, self.op, self.terms)

    def __mul__(self, other):  # `k1 * k2` -> KernelProduct; `k * 0.5` -> ScaledKernel
        if isinstance(other, Kernel):
            return Kernel._combine(2, self, other)
        return self.__rmul__(other)

    def _transform_single(self, t) -> "Kernel":
        if isinstance(t, ARDTransform):
            v = tuple(float(a) for a in t.v)
            if self.ard is not None:
                if len(self.ard) != len(v):
                    raise ValueError("ARDTransform dimensions do not match")
                v = tuple(a * b for a, b in zip(self.ard, v))
            return Kernel(self.kind, self.variance, self.inv_lengthscale, v, self.param)
        return Kernel(self.kind, self.variance, self.inv_lengthscale * t.s, self.ard, self.param)

    def compose(self, t) -> "Kernel":
        """`k ∘ ScaleTransform(s)` / `k ∘ ARDTransform(v)`: inputs are scaled before distances are taken; the transform of a
        KernelSum / KernelProduct feeds every term."""
        return Kernel._from_terms(self.op, tuple(k._transform_single(t) for k in self.all_terms()))

    __matmul__ = compose


@dataclass(frozen=True)
class ScaleTransform:
    s: float


class ARDTransform:
    """KernelFunctions `ARDTransform(v)`: x -> v .* x (one positive multiplier per input dimension, D <= 8)."""

    def __init__(self, v):
        self.v = tuple(float(a) for a in np.asarray(v, dtype=np.float64).reshape(-1))


def SEKernel() -> Kernel:
    return Kernel(0)


SqExponentialKernel = SEKernel


def Matern32Kernel() -> Kernel:
    return Kernel(1)


def Matern52Kernel() -> Kernel:
    return Kernel(2)


def ExponentialKernel() -> Kernel:  # KernelFunctions: ExponentialKernel == Matern12Kernel, κ(d) = exp(-d)
    return Kernel(3)


Matern12Kernel = ExponentialKernel


def RationalQuadraticKernel(alpha: float = 2.0) -> Kernel:  # κ(d²) = (1 + d²/(2α))^(-α)
    if not alpha > 0:
        raise ValueError("RationalQuadraticKernel needs α > 0")
    return Kernel(4, param=float(alpha))


def PeriodicKernel(r: float = 1.0) -> Kernel:
    """KernelFunctions `PeriodicKernel(; r)`: κ = exp(-0.5 Σ_k (sinpi(x_k - x'_k) / r)²) (metric `Sinus(r)`), one r for all dimensions."""
    if not r > 0:
        raise ValueError("PeriodicKernel needs r > 0")
    return Kernel(5, param=float(r))


def with_lengthscale(k: Kernel, l: float) -> Kernel:
    return k.compose(ScaleTransform(1.0 / float(l)))


class AbstractGP:
    def __call__(self, x, sigma2=1e-18):
        return FiniteGP(self, x, sigma2)


class GP(AbstractGP):
    """`GP(kernel)` (zero mean) or `GP(c, kernel)` (constant mean c)."""

    def __init__(self, *args):
        if len(args) == 1:
            self.mean_const, self.kernel = 0.0, args[0]
        elif len(args) == 2:
            self.mean_const, self.kernel = float(args[0]), args[1]
        else:
            raise TypeError("GP(kernel) or GP(mean_const, kernel)")
        if not isinstance(self.kernel, Kernel):
            raise TypeError("unsupported kernel type (liblmm supports SE / Matern32 / Matern52 / Exponential / RationalQuadratic / Periodic, scaled, stretched, summed or multiplied)")

    def __eq__(self, other):
        return isinstance(other, GP) and (self.mean_const, self.kernel) == (other.mean_const, other.kernel)

    def __hash__(self):
        return hash((self.mean_const, self.kernel))


class ColVecs:
    """D x N matrix whose columns are the inputs."""

    def __init__(self, X):
        self.X = np.asarray(X, dtype=np.float64)

    def points(self) -> np.ndarray:  # (N, D) C-order == D x N column-major
        return np.ascontiguousarray(self.X.T)


class RowVecs:
    """N x D matrix whose rows are the inputs."""

    def __init__(self, X):
        self.X = np.asarray(X, dtype=np.float64)

    def points(self) -> np.ndarray:
        return np.ascontiguousarray(self.X)


def _points(x) -> np.ndarray:
    """(N, D) C-contiguous float64 view of a Vector{<:Real} / ColVecs / RowVecs input."""
    if isinstance(x, (ColVecs, RowVecs)):
        return x.points()
    if _is_device_tensor(x):
        return x
    a = np.asarray(x, dtype=np.float64)
    if a.ndim != 1:
        raise TypeError("inputs must be a real vector, ColVecs or RowVecs")
    return np.ascontiguousarray(a.reshape(-1, 1))


def _is_device_tensor(a) -> bool:
    return hasattr(a, "data_ptr") and getattr(a, "is_cuda", False)


class MOInputIsotopicByOutputs:
    """Element (j-1)N + i is (x[i], j)."""

    def __init__(self, x, out_dim: int):
        self.x = x
        self.out_dim = int(out_dim)

    def __len__(self):
        return _npoints(self.x) * self.out_dim


class MOInputIsotopicByFeatures:
    """Element (i-1)p + j is (x[i], j)."""

    def __init__(self, x, out_dim: int):
        self.x = x
        self.out_dim = int(out_dim)

    def __len__(self):
        return _npoints(self.x) * self.out_dim


def _npoints(x) -> int:
    p = _points(x)
    return int(p.shape[0])


def indices_which_reorder_outputs_to_features(x) -> np.ndarray:
    """src/independent_mogp.jl:135-139 (0-based)."""
    out = np.zeros(len(x), dtype=np.int64)
    _lib.load().lmm_reorder_indices(_npoints(x.x), x.out_dim, 0, out.ctypes.data_as(C.c_void_p))
    return out


def indices_which_reorder_features_to_outputs(x) -> np.ndarray:
    """src/independent_mogp.jl:141-145 (0-based)."""
    out = np.zeros(len(x), dtype=np.int64)
    _lib.load().lmm_reorder_indices(_npoints(x.x), x.out_dim, 1, out.ctypes.data_as(C.c_void_p))
    return out


# --------------------------------------------------------------------------------------------
# models (src/LinearMixingModels.jl:21-24 exports)
# --------------------------------------------------------------------------------------------
class Orthogonal:
    """`Orthogonal(U, S; validate_fields=true)`: H = U * sqrt(S)  (src/orthogonal_matrix.jl:11-19)."""

    def __init__(self, U, S, validate_fields: bool = True):
        U = np.asarray(U, dtype=np.float64)
        S = np.asarray(S, dtype=np.float64)
        if S.ndim == 2:  # Diagonal(S) given as a matrix
            S = np.diag(S).copy()
        if U.ndim != 2 or S.ndim != 1 or U.shape[1] != S.shape[0]:
            raise TypeError("Orthogonal(U::Matrix p x m, S::Diagonal m x m)")
        self.U = np.asfortranarray(U)
        self.S = np.ascontiguousarray(S)
        if validate_fields:
            rc = _lib.load().lmm_orthogonal_validate(ptr(self.U), U.shape[0], U.shape[1])
            if rc == _lib.LMM_E_NOT_ORTHOGONAL:
                raise ValueError("`U` is not an orthogonal matrix")  # ArgumentError, src/orthogonal_matrix.jl:22

    @property
    def shape(self):
        return self.U.shape

    def __array__(self, dtype=None, copy=None):  # collect(H)
        return self.U * np.sqrt(self.S)[None, :]


class IndependentMOGP(AbstractGP):
    """src/independent_mogp.jl:10-12."""

    def __init__(self, fs: Sequence[AbstractGP]):
        fs = list(fs)
        if not fs or not all(isinstance(f, (GP, PosteriorGP)) for f in fs):
            raise TypeError("IndependentMOGP(fs::Vector{<:AbstractGP})")
        self.fs = fs


def independent_mogp(fs) -> IndependentMOGP:
    return IndependentMOGP(fs)


class ILMM(AbstractGP):
    """src/ilmm.jl:16-19.  `OILMM` is the case H::Orthogonal with IndependentMOGP latents."""

    def __init__(self, f: AbstractGP, H):
        if not isinstance(f, AbstractGP):
            raise TypeError("ILMM(f::AbstractGP, H::AbstractMatrix)")
        self.f = f
        self.H = H if isinstance(H, Orthogonal) else np.asfortranarray(np.asarray(H, dtype=np.float64))
        if not isinstance(H, Orthogonal) and self.H.ndim != 2:
            raise TypeError("H must be a matrix")


class _OILMMMeta(type):
    def __instancecheck__(cls, obj):
        return isinstance(obj, ILMM) and isinstance(obj.f, IndependentMOGP) and isinstance(obj.H, Orthogonal)


class OILMM(metaclass=_OILMMMeta):
    """`const OILMM = ILMM{<:IndependentMOGP,<:Orthogonal}` (src/oilmm.jl:13): usable in isinstance."""

    def __new__(cls, fs, H):
        f = fs if isinstance(fs, IndependentMOGP) else IndependentMOGP(fs)
        if not isinstance(H, Orthogonal):
            raise TypeError("OILMM needs an Orthogonal mixing matrix")
        return ILMM(f, H)


def get_latent_gp(f: ILMM):
    return f.f


class PosteriorGP(AbstractGP):
    """View of one latent `PosteriorGP(prior, (α, C, x, δ))` held on the device."""

    def __init__(self, owner: "_PostHandle", index: int, prior: GP):
        self._owner, self.index, self.prior = owner, index, prior

    def _export(self, want_L=False):
        return self._owner.export(self.index, want_L)

    @property
    def alpha(self):
        return self._export()[1]

    @property
    def delta(self):
        return self._export()[2]

    @property
    def C(self):
        """Lower Cholesky factor L of K + Σ (C.L in Julia)."""
        return self._export(True)[0]


class _PostHandle:
    """Owns an `lmm_post*`."""

    def __init__(self, ctx: Context, handle, N: int, joint_n: int = 0):
        self.ctx, self.handle, self.N, self.joint_n = ctx, handle, N, joint_n
        self._finalizer = weakref.finalize(self, ctx.lib.lmm_post_free, handle)

    def free(self):
        self._finalizer()

    def export(self, i: int, want_L: bool):
        n = self.joint_n or self.N
        L = np.zeros((n, n), order="F") if want_L else None
        a, d = np.zeros(n), np.zeros(n)
        rc = self.ctx.lib.lmm_post_export(self.handle, i, ptr(L), ptr(a), ptr(d))
        self.ctx.check(rc)
        return L, a, d

    def device_bytes(self) -> int:
        b = C.c_int64()
        self.ctx.lib.lmm_post_info(self.handle, None, None, None, None, None, C.byref(b))
        return b.value


class _JointPosterior(AbstractGP):
    """`PosteriorGP{IndependentMOGP}`: joint (mN) posterior of a general ILMM (src/ilmm.jl:196)."""

    def __init__(self, owner: _PostHandle, prior: IndependentMOGP):
        self._owner, self.prior = owner, prior


# --------------------------------------------------------------------------------------------
# FiniteGP and the AbstractGPs verbs
# --------------------------------------------------------------------------------------------
@dataclass
class Normal:
    mu: float
    sigma: float


class FiniteGP:
    """`f(x, σ²)` -- AbstractGPs: a scalar gives `Diagonal(Fill(σ², n))` (the reference's fast paths), a vector
    `Diagonal(v)`, a matrix a dense Σy.  Non-scalar noise is only defined for an IndependentMOGP (the
    AbstractGPs generic FiniteGP path, test/independent_mogp.jl:72-75); ILMM / OILMM methods dispatch on
    scalar noise only (src/ilmm.jl:45) and raise TypeError otherwise, as the reference's MethodError does."""

    def __init__(self, f: AbstractGP, x, sigma2=1e-18):
        self.f, self.x = f, x
        self.noise = None  # ndarray (1-D: diagonal, 2-D: dense), in the ordering of `x`
        if isinstance(sigma2, (int, float, np.floating)):
            self.sigma2 = float(sigma2)
        else:
            a = np.asarray(sigma2, dtype=np.float64)
            n = len(x)
            if a.ndim not in (1, 2) or a.shape[0] != n or (a.ndim == 2 and a.shape[1] != n):
                raise ValueError("observation noise must be a scalar, a length-n vector or an n x n matrix")
            if isinstance(f, ILMM):
                raise TypeError("ILMM / OILMM methods need scalar observation noise (src/ilmm.jl:45)")
            self.noise = a
            self.sigma2 = 0.0

    def __len__(self):
        return len(self.x)


def noise_var(fx: FiniteGP) -> float:
    """src/ilmm.jl:41."""
    return fx.sigma2


def reshape_y(y, N: int) -> np.ndarray:
    """src/ilmm.jl:43: `reshape(y, N, :)'` (p x N)."""
    return np.asarray(y).reshape(-1, N)


def unpack(fx: FiniteGP):
    """src/ilmm.jl:45-54."""
    if not (isinstance(fx.f, ILMM) and isinstance(fx.x, MOInputIsotopicByOutputs)):
        raise TypeError("unpack(fx::FiniteGP{<:ILMM,<:MOInputIsotopicByOutputs,<:Diagonal{<:Real,<:Fill}})")
    H = fx.f.H
    if fx.x.out_dim != H.shape[0]:
        raise RuntimeError("out dim of x != out dim of f.")
    return fx.f.f, H, fx.sigma2, fx.x.x


def _descs(fs: Sequence[GP]):
    arr = (GpDesc * len(fs))()
    keep = []  # the ARD / extra-term arrays must outlive the call; they ride on the ctypes array

    def ard_ptr(k):
        if k.ard is None:
            return None
        a = np.ascontiguousarray(k.ard, dtype=np.float64)
        keep.append(a)
        return a.ctypes.data

    for i, f in enumerate(fs):
        g = f.prior if isinstance(f, PosteriorGP) else f
        k = g.kernel
        extra, n_extra = None, len(k.terms)
        if n_extra:
            ex = (_lib.KernelTerm * n_extra)()
            for t, q in enumerate(k.terms):
                ex[t] = _lib.KernelTerm(q.kind, 0, q.variance, q.inv_lengthscale, q.param, ard_ptr(q))
            keep.append(ex)
            extra = C.cast(ex, C.c_void_p)
        arr[i] = GpDesc(k.kind, k.op if n_extra else 0, k.variance, k.inv_lengthscale, g.mean_const, ard_ptr(k), k.param, n_extra, 0, extra)
    arr._keep = keep
    return arr


def _yvec(y, n: int):
    if _is_device_tensor(y):
        if y.numel() != n:
            raise ValueError("length of y does not match the inputs")
        return y
    a = np.ascontiguousarray(np.asarray(y, dtype=np.float64).reshape(-1))
    if a.shape[0] != n:
        raise ValueError("length of y does not match the inputs")
    return a


def _ctx_of(fx: FiniteGP) -> Context:
    f = fx.f
    owner = None
    if isinstance(f, ILMM):
        lat = f.f
        if isinstance(lat, IndependentMOGP) and isinstance(lat.fs[0], PosteriorGP):
            owner = lat.fs[0]._owner
        elif isinstance(lat, _JointPosterior):
            owner = lat._owner
    elif isinstance(f, IndependentMOGP) and isinstance(f.fs[0], PosteriorGP):
        owner = f.fs[0]._owner
    elif isinstance(f, (_JointPosterior, _MissingDataPosterior)):
        owner = f._owner
    return owner.ctx if owner is not None else default_context()


def _post_owner(fx: FiniteGP) -> Optional[_PostHandle]:
    f = fx.f
    lat = f.f if isinstance(f, ILMM) else f
    if isinstance(lat, IndependentMOGP) and isinstance(lat.fs[0], PosteriorGP):
        return lat.fs[0]._owner
    if isinstance(lat, (_JointPosterior, _MissingDataPosterior)):
        return lat._owner
    return None


def _noise_by_outputs(fx: FiniteGP):
    """(kind, Σy in by-outputs order) for a FiniteGP with non-scalar noise: kind 1 diagonal, 2 dense
    (src/independent_mogp.jl:149-151 `reorder_by_outputs(Σy, x)`)."""
    a = fx.noise
    if isinstance(fx.x, MOInputIsotopicByFeatures):
        idx = indices_which_reorder_features_to_outputs(fx.x)
        a = a[idx] if a.ndim == 1 else a[np.ix_(idx, idx)]
    return (1, np.ascontiguousarray(a)) if a.ndim == 1 else (2, np.asfortranarray(a))


def _add_noise_to_var(fx: FiniteGP, V: np.ndarray) -> np.ndarray:
    return V if fx.noise is None else V + (fx.noise if fx.noise.ndim == 1 else np.diag(fx.noise))


def _require_by_outputs(fx: FiniteGP):
    if not isinstance(fx.x, MOInputIsotopicByOutputs):
        raise TypeError("this method needs MOInputIsotopicByOutputs inputs (src/ilmm.jl:45)")


def logpdf(fx: FiniteGP, y):
    """`logpdf(fx, y)`: src/oilmm.jl:79-93, src/ilmm.jl:150-163, src/independent_mogp.jl:74-80,222-229.
    A matrix `Y` (one sample per column, as returned by `rand(rng, fx, n)`) gives the vector of
    per-column logpdfs (AbstractGPs `logpdf(fx, Y::AbstractMatrix)`)."""
    if not _is_device_tensor(y):
        ya = np.asarray(y)
        if ya.ndim == 2:
            return np.array([_logpdf_impl(fx, np.ascontiguousarray(ya[:, k]))[0] for k in range(ya.shape[1])])
    return _logpdf_impl(fx, y)[0]


def logpdf_terms(fx: FiniteGP, y) -> np.ndarray:
    """Per-latent lml terms followed by the regulariser (OILMM / IndependentMOGP)."""
    return _logpdf_impl(fx, y)[1]


def _logpdf_impl(fx: FiniteGP, y):
    f = fx.f
    ctx = _ctx_of(fx)
    lib = ctx.lib
    out = C.c_double()
    il = C.c_int(-1)
    owner = _post_owner(fx)
    if fx.noise is not None and (owner is not None or not isinstance(f, IndependentMOGP)):
        # AbstractGPs generic `logpdf(fx, y)` on (mean, cov + Σy), e.g. a posterior evaluated under a vector / dense Σy
        M, Cm = mean_and_cov(fx)
        yv = _yvec(y, M.shape[0])
        Cf = np.asfortranarray(Cm)
        rc = lib.lmm_mvn_logpdf_rand(ctx.handle, ptr(M), ptr(Cf), M.shape[0], ptr(yv), C.byref(out), None, None, C.byref(il))
        ctx.check(rc)
        return out.value, None
    if isinstance(f, IndependentMOGP) and isinstance(fx.x, MOInputIsotopicByFeatures):
        # src/independent_mogp.jl:222-229
        xo = MOInputIsotopicByOutputs(fx.x.x, fx.x.out_dim)
        idx = indices_which_reorder_features_to_outputs(fx.x)
        noise = fx.sigma2 if fx.noise is None else _noise_by_outputs(fx)[1]
        return _logpdf_impl(FiniteGP(f, xo, noise), np.asarray(y, dtype=np.float64)[idx])
    _require_by_outputs(fx)
    pts = _points(fx.x.x)
    N, D = int(pts.shape[0]), int(pts.shape[1])
    if fx.noise is not None:
        kind, Sy = _noise_by_outputs(fx)
        yv = _yvec(y, N * fx.x.out_dim)
        rc = lib.lmm_imogp_posterior_noise(ctx.handle, _descs(f.fs), len(f.fs), ptr(pts), N, D, ptr(Sy), kind, ptr(yv), fx.x.out_dim, None,
                                           C.byref(out), C.byref(il))
        ctx.check(rc, il.value)
        return out.value, None
    if owner is not None:
        if isinstance(f, ILMM) and f.H.shape[0] != fx.x.out_dim:
            raise RuntimeError("out dim of x != out dim of f.")
        yv = _yvec(y, N * fx.x.out_dim)
        rc = lib.lmm_post_logpdf(owner.handle, ptr(pts), N, fx.sigma2, ptr(yv), C.byref(out), C.byref(il))
        ctx.check(rc, il.value)
        return out.value, None
    if isinstance(f, ILMM):
        lat, H, s2, _ = unpack(fx)
        if not isinstance(lat, IndependentMOGP):
            raise TypeError("ILMM latents must be an IndependentMOGP")
        m = len(lat.fs)
        yv = _yvec(y, N * fx.x.out_dim)
        if isinstance(H, Orthogonal):
            terms = np.zeros(m + 1)
            rc = lib.lmm_oilmm_logpdf(ctx.handle, _descs(lat.fs), m, ptr(pts), N, D, ptr(H.U), ptr(H.S), H.shape[0], s2, ptr(yv),
                                      fx.x.out_dim, C.byref(out), ptr(terms), C.byref(il))
            ctx.check(rc, il.value)
            return out.value, terms
        rc = lib.lmm_ilmm_logpdf(ctx.handle, _descs(lat.fs), m, ptr(pts), N, D, ptr(H), H.shape[0], s2, ptr(yv), fx.x.out_dim,
                                 _lib_ilmm_form(), C.byref(out), C.byref(il))
        ctx.check(rc, il.value)
        return out.value, None
    if isinstance(f, IndependentMOGP):
        m = len(f.fs)
        yv = _yvec(y, N * fx.x.out_dim)
        terms = np.zeros(m + 1)
        rc = lib.lmm_imogp_logpdf(ctx.handle, _descs(f.fs), m, ptr(pts), N, D, fx.sigma2, ptr(yv), fx.x.out_dim, C.byref(out),
                                  ptr(terms), C.byref(il))
        ctx.check(rc, il.value)
        return out.value, terms
    raise TypeError(f"logpdf not defined for FiniteGP of {type(f).__name__}")


_ILMM_FORM = 0


def _lib_ilmm_form() -> int:
    return _ILMM_FORM


def set_ilmm_form(form: int) -> None:
    """0: the reference's projected (mN) form; 1: dense pN form H K H' + σ²I (test oracle form)."""
    global _ILMM_FORM
    _ILMM_FORM = int(form)


def posterior(fx: FiniteGP, y, with_logpdf: bool = False):
    """`posterior(fx, y)`: src/oilmm.jl:116-134, src/ilmm.jl:184-198, src/independent_mogp.jl:119-126.
    `with_logpdf=True` additionally returns logpdf(fx, y) from the same factorisation."""
    f = fx.f
    ctx = _ctx_of(fx)
    lib = ctx.lib
    if isinstance(f, IndependentMOGP) and isinstance(fx.x, MOInputIsotopicByFeatures):
        # AbstractGPs generic posterior on by-features inputs == the by-outputs posterior of the reordered data
        xo = MOInputIsotopicByOutputs(fx.x.x, fx.x.out_dim)
        idx = indices_which_reorder_features_to_outputs(fx.x)
        noise = fx.sigma2 if fx.noise is None else _noise_by_outputs(fx)[1]
        return posterior(FiniteGP(f, xo, noise), np.asarray(y, dtype=np.float64)[idx], with_logpdf)
    _require_by_outputs(fx)
    pts = _points(fx.x.x)
    N, D = int(pts.shape[0]), int(pts.shape[1])
    h = C.c_void_p()
    out = C.c_double()
    il = C.c_int(-1)
    lp = C.byref(out) if with_logpdf else None
    owner0 = _post_owner(fx)
    if fx.noise is not None:
        if owner0 is not None or not isinstance(f, IndependentMOGP):
            raise NotImplementedError("non-scalar observation noise is built for IndependentMOGP priors")
        kind, Sy = _noise_by_outputs(fx)
        m = len(f.fs)
        yv = _yvec(y, N * fx.x.out_dim)
        rc = lib.lmm_imogp_posterior_noise(ctx.handle, _descs(f.fs), m, ptr(pts), N, D, ptr(Sy), kind, ptr(yv), fx.x.out_dim, C.byref(h), lp,
                                           C.byref(il))
        ctx.check(rc, il.value)
        if kind == 1:
            owner = _PostHandle(ctx, h, N)
            post = IndependentMOGP([PosteriorGP(owner, i, g) for i, g in enumerate(f.fs)])
        else:  # dense Σy couples the outputs: one joint PosteriorGP{IndependentMOGP}
            post = _JointPosterior(_PostHandle(ctx, h, N, joint_n=m * N), f)
        return (post, out.value) if with_logpdf else post
    if owner0 is not None:
        # sequential conditioning: posterior(post(x2, σ²), y2)
        if isinstance(f, ILMM) and f.H.shape[0] != fx.x.out_dim:
            raise RuntimeError("out dim of x != out dim of f.")
        lat = f.f if isinstance(f, ILMM) else f
        yv = _yvec(y, N * fx.x.out_dim)
        logp = logpdf(fx, y) if with_logpdf else None
        rc = lib.lmm_post_condition(owner0.handle, ptr(pts), N, fx.sigma2, ptr(yv), C.byref(h), C.byref(il))
        ctx.check(rc, il.value)
        if isinstance(lat, _JointPosterior):  # general ILMM: src/ilmm.jl:184-198 on PosteriorGP{IndependentMOGP} latents
            m = len(lat.prior.fs)
            owner = _PostHandle(ctx, h, owner0.N + N, joint_n=m * (owner0.N + N))
            post = ILMM(_JointPosterior(owner, lat.prior), f.H)
            return (post, logp) if with_logpdf else post
        owner = _PostHandle(ctx, h, owner0.N + N)
        newlat = IndependentMOGP([PosteriorGP(owner, i, g.prior) for i, g in enumerate(lat.fs)])
        post = ILMM(newlat, f.H) if isinstance(f, ILMM) else newlat
        return (post, logp) if with_logpdf else post
    if isinstance(f, ILMM):
        lat, H, s2, _ = unpack(fx)
        if not isinstance(lat, IndependentMOGP):
            raise TypeError("ILMM latents must be an IndependentMOGP")
        m = len(lat.fs)
        yv = _yvec(y, N * fx.x.out_dim)
        if isinstance(H, Orthogonal):
            rc = lib.lmm_oilmm_posterior(ctx.handle, _descs(lat.fs), m, ptr(pts), N, D, ptr(H.U), ptr(H.S), H.shape[0], s2, ptr(yv),
                                         fx.x.out_dim, C.byref(h), lp, None, C.byref(il))
            ctx.check(rc, il.value)
            owner = _PostHandle(ctx, h, N)
            post = ILMM(IndependentMOGP([PosteriorGP(owner, i, g) for i, g in enumerate(lat.fs)]), H)
        else:
            rc = lib.lmm_ilmm_posterior(ctx.handle, _descs(lat.fs), m, ptr(pts), N, D, ptr(H), H.shape[0], s2, ptr(yv), fx.x.out_dim,
                                        C.byref(h), lp, C.byref(il))
            ctx.check(rc, il.value)
            owner = _PostHandle(ctx, h, N, joint_n=m * N)
            post = ILMM(_JointPosterior(owner, lat), H)
    elif isinstance(f, IndependentMOGP):
        m = len(f.fs)
        yv = _yvec(y, N * fx.x.out_dim)
        rc = lib.lmm_imogp_posterior(ctx.handle, _descs(f.fs), m, ptr(pts), N, D, fx.sigma2, ptr(yv), fx.x.out_dim, C.byref(h), lp,
                                     C.byref(il))
        ctx.check(rc, il.value)
        owner = _PostHandle(ctx, h, N)
        post = IndependentMOGP([PosteriorGP(owner, i, g) for i, g in enumerate(f.fs)])
    else:
        raise TypeError(f"posterior not defined for FiniteGP of {type(f).__name__}")
    return (post, out.value) if with_logpdf else post


def mean_and_var(fx: FiniteGP) -> Tuple[np.ndarray, np.ndarray]:
    """`mean_and_var(fx)`: src/oilmm.jl:57-76, src/ilmm.jl:122-129, src/independent_mogp.jl:50-57."""
    f = fx.f
    if isinstance(f, PosteriorGP):
        # one latent of a posterior on its own, `mean_and_var(get_latent_gp(post).fs[i](x*, σ²))` -- the per-latent
        # call src/oilmm.jl:61 makes (AbstractGPs FiniteGP{<:PosteriorGP})
        pts = _points(fx.x)
        Ns = int(pts.shape[0])
        M, V = np.zeros(Ns), np.zeros(Ns)
        c = f._owner.ctx
        c.check(c.lib.lmm_post_latent_mean_and_var(f._owner.handle, f.index, ptr(pts), Ns, fx.sigma2, ptr(M), ptr(V)))
        return M, V
    if isinstance(f, GP):  # AbstractGPs `mean_and_var(f(x, σ²))` for a prior GP: (m(x), diag K + σ²)
        Ns = _npoints(fx.x)
        return np.full(Ns, f.mean_const), np.full(Ns, f.kernel.kdiag + fx.sigma2)
    owner = _post_owner(fx)
    needs_device = owner is not None or isinstance(f, ILMM)
    ctx = _ctx_of(fx) if needs_device else None
    lib = ctx.lib if ctx else None
    x = fx.x
    reorder = None
    if isinstance(f, (IndependentMOGP, _JointPosterior)) and isinstance(x, MOInputIsotopicByFeatures):
        reorder = indices_which_reorder_outputs_to_features(x)  # src/independent_mogp.jl:169-179
        x = MOInputIsotopicByOutputs(x.x, x.out_dim)
    elif not isinstance(x, MOInputIsotopicByOutputs):
        raise TypeError("this method needs MOInput inputs")
    pts = _points(x.x)
    Ns, D = int(pts.shape[0]), int(pts.shape[1])
    p = x.out_dim
    M, V = np.zeros(p * Ns), np.zeros(p * Ns)
    if isinstance(f, ILMM) and f.H.shape[0] != p:
        raise RuntimeError("out dim of x != out dim of f.")
    if owner is not None:
        rc = lib.lmm_post_mean_and_var(owner.handle, ptr(pts), Ns, fx.sigma2, ptr(M), ptr(V))
        ctx.check(rc)
    elif isinstance(f, ILMM):
        lat, H = f.f, f.H
        m = len(lat.fs)
        if isinstance(H, Orthogonal):
            rc = lib.lmm_oilmm_prior_mean_and_var(ctx.handle, _descs(lat.fs), m, ptr(pts), Ns, D, ptr(H.U), ptr(H.S), p, fx.sigma2, p,
                                                  ptr(M), ptr(V))
        else:
            rc = lib.lmm_ilmm_prior_mean_and_var(ctx.handle, _descs(lat.fs), m, ptr(pts), Ns, D, ptr(H), p, fx.sigma2, p, ptr(M), ptr(V))
        ctx.check(rc)
    elif isinstance(f, IndependentMOGP):
        if len(f.fs) != p:
            raise RuntimeError("out dim of x != out dim of f.")
        # prior: mean const, var = variance + σ² (src/independent_mogp.jl:50-57); trivial, no kernel needed
        M = np.concatenate([np.full(Ns, g.mean_const) for g in f.fs])
        V = np.concatenate([np.full(Ns, g.kernel.kdiag + fx.sigma2) for g in f.fs])
    else:
        raise TypeError(f"mean_and_var not defined for FiniteGP of {type(f).__name__}")
    if reorder is not None:
        M, V = M[reorder], V[reorder]
    return M, _add_noise_to_var(fx, V)


def mean_and_cov(fx: FiniteGP) -> Tuple[np.ndarray, np.ndarray]:
    """`mean_and_cov(fx)`: src/ilmm.jl:132-139 (also the path `cov(fx::FiniteGP{<:OILMM})` takes),
    src/independent_mogp.jl:60-63 + Σy.  Dense (p N*)² output -- meant for small N*."""
    f = fx.f
    ctx = _ctx_of(fx)
    owner = _post_owner(fx)
    x = fx.x
    reorder = None
    if isinstance(f, (IndependentMOGP, _JointPosterior)) and isinstance(x, MOInputIsotopicByFeatures):
        reorder = indices_which_reorder_outputs_to_features(x)  # src/independent_mogp.jl:181-186
        x = MOInputIsotopicByOutputs(x.x, x.out_dim)
    elif not isinstance(x, MOInputIsotopicByOutputs):
        raise TypeError("this method needs MOInput inputs")
    pts = _points(x.x)
    Ns, D = int(pts.shape[0]), int(pts.shape[1])
    p = x.out_dim
    if isinstance(f, ILMM) and f.H.shape[0] != p:
        raise RuntimeError("out dim of x != out dim of f.")
    M = np.zeros(p * Ns)
    Cm = np.zeros((p * Ns, p * Ns), order="F")
    if owner is not None:
        rc = ctx.lib.lmm_post_mean_and_cov(owner.handle, ptr(pts), Ns, fx.sigma2, ptr(M), ptr(Cm))
    else:
        if isinstance(f, ILMM):
            fs, H, jitter = f.f.fs, np.asfortranarray(np.asarray(f.H, dtype=np.float64)), 1e-18
        elif isinstance(f, IndependentMOGP):
            if len(f.fs) != p:
                raise RuntimeError("out dim of x != out dim of f.")
            fs, H, jitter = f.fs, np.asfortranarray(np.eye(p)), 0.0
        else:
            raise TypeError(f"mean_and_cov not defined for FiniteGP of {type(f).__name__}")
        rc = ctx.lib.lmm_prior_mean_and_cov(ctx.handle, _descs(fs), len(fs), ptr(pts), Ns, D, ptr(H), p, fx.sigma2, jitter, p, ptr(M), ptr(Cm))
    ctx.check(rc)
    Cm = np.ascontiguousarray(Cm)
    if reorder is not None:
        M, Cm = M[reorder], Cm[np.ix_(reorder, reorder)]
    if fx.noise is not None:
        Cm = Cm + (np.diag(fx.noise) if fx.noise.ndim == 1 else fx.noise)
    return M, Cm


def cov(*args) -> np.ndarray:
    """`cov(fx)` (src/ilmm.jl:147) or, for an IndependentMOGP prior, the process cross-covariance
    `cov(f, x, y)` between two isotopic inputs in any by-outputs / by-features combination
    (src/independent_mogp.jl:60-71, 181-215; test/independent_mogp.jl:135-141)."""
    if len(args) == 1:
        return mean_and_cov(args[0])[1]
    f, x = args[0], args[1]
    y = args[2] if len(args) > 2 else x
    if not isinstance(f, IndependentMOGP) or any(isinstance(g, PosteriorGP) for g in f.fs):
        raise TypeError("cov(f, x[, y]) is built for IndependentMOGP priors")
    for z in (x, y):
        if not isinstance(z, (MOInputIsotopicByOutputs, MOInputIsotopicByFeatures)) or z.out_dim != len(f.fs):
            raise TypeError("cov(f, x, y) needs isotopic multi-output inputs with out_dim == number of outputs")
    ctx = default_context()
    pa, pb = _points(x.x), _points(y.x)
    m, Na, Nb = len(f.fs), int(pa.shape[0]), int(pb.shape[0])
    out = np.zeros((m * Na, m * Nb), order="F")
    rc = ctx.lib.lmm_imogp_cross_cov(ctx.handle, _descs(f.fs), m, ptr(pa), Na, ptr(pb), Nb, int(pa.shape[1]), ptr(out))
    ctx.check(rc)
    out = np.ascontiguousarray(out)
    if isinstance(x, MOInputIsotopicByFeatures):
        out = out[indices_which_reorder_outputs_to_features(x), :]
    if isinstance(y, MOInputIsotopicByFeatures):
        out = out[:, indices_which_reorder_outputs_to_features(y)]
    return out


def mean(fx: FiniteGP) -> np.ndarray:
    return mean_and_var(fx)[0]  # src/ilmm.jl:142


def var(fx: FiniteGP) -> np.ndarray:
    return mean_and_var(fx)[1]  # src/ilmm.jl:145


def marginals(fx: FiniteGP) -> List[Normal]:
    """AbstractGPs generic: `Normal.(m, sqrt.(v))`."""
    M, V = mean_and_var(fx)
    return [Normal(float(a), math.sqrt(float(b))) for a, b in zip(M, V)]


def rand(*args):
    """`rand([rng,] fx[, n_samples])`: src/oilmm.jl:40-54, src/ilmm.jl:78-106, src/independent_mogp.jl:83-99.
    Standard normals are drawn on the host from `rng` in the reference's order (latent 1..m, N each;
    then p*N noise draws) and handed to the library, so a sample is a deterministic function of them."""
    args = list(args)
    rng = args.pop(0) if isinstance(args[0], np.random.Generator) else np.random.default_rng()
    fx = args.pop(0)
    if args:
        return np.stack([_rand_one(rng, fx) for _ in range(int(args[0]))], axis=1)  # src/ilmm.jl:90-92
    return _rand_one(rng, fx)


def _rand_one(rng, fx: FiniteGP) -> np.ndarray:
    f = fx.f
    ctx = _ctx_of(fx)
    lib = ctx.lib
    owner = _post_owner(fx)
    by_features = isinstance(f, (IndependentMOGP, _JointPosterior)) and isinstance(fx.x, MOInputIsotopicByFeatures)
    if not by_features:
        _require_by_outputs(fx)
    pts = _points(fx.x.x)
    N, D = int(pts.shape[0]), int(pts.shape[1])
    p = fx.x.out_dim
    il = C.c_int(-1)
    out = np.zeros(p * N)
    if fx.noise is not None:
        # AbstractGPs generic `rand(rng, fx) = m + cholesky(K + Σy).U' z`: covariance and factor on the device
        M, Cm = mean_and_cov(fx)
        Cf, z = np.asfortranarray(Cm), rng.standard_normal(p * N)
        rc = lib.lmm_mvn_logpdf_rand(ctx.handle, ptr(M), ptr(Cf), p * N, None, None, ptr(z), ptr(out), C.byref(il))
        ctx.check(rc)
        return out
    if isinstance(f, _MissingDataPosterior):
        if f.prior.H.shape[0] != p:
            raise RuntimeError("out dim of x != out dim of f.")
        z = rng.standard_normal(p * N)
        rc = lib.lmm_post_rand(owner.handle, ptr(pts), N, fx.sigma2, ptr(z), None, ptr(out), C.byref(il))
        ctx.check(rc, il.value)
        return out
    if isinstance(f, _JointPosterior):
        z = rng.standard_normal(p * N)
        rc = lib.lmm_post_rand(owner.handle, ptr(pts), N, fx.sigma2, ptr(z), None, ptr(out), C.byref(il))
        ctx.check(rc, il.value)
        return out.reshape(p, N).T.reshape(-1).copy() if by_features else out
    if isinstance(f, ILMM):
        if f.H.shape[0] != p:
            raise RuntimeError("out dim of x != out dim of f.")
        m = f.H.shape[1]
        z_lat = rng.standard_normal(m * N)
        z_noise = rng.standard_normal(p * N)
        if owner is not None:
            rc = lib.lmm_post_rand(owner.handle, ptr(pts), N, fx.sigma2, ptr(z_lat), ptr(z_noise), ptr(out), C.byref(il))
        elif isinstance(f.H, Orthogonal):
            rc = lib.lmm_oilmm_rand(ctx.handle, _descs(f.f.fs), m, ptr(pts), N, D, ptr(f.H.U), ptr(f.H.S), p, fx.sigma2, p, ptr(z_lat),
                                    ptr(z_noise), ptr(out), C.byref(il))
        else:
            rc = lib.lmm_ilmm_rand(ctx.handle, _descs(f.f.fs), m, ptr(pts), N, D, ptr(f.H), p, fx.sigma2, p, ptr(z_lat), ptr(z_noise),
                                   ptr(out), C.byref(il))
        ctx.check(rc, il.value)
        return out
    if isinstance(f, IndependentMOGP):
        m = len(f.fs)
        z = rng.standard_normal(m * N)
        if owner is not None:
            rc = lib.lmm_post_rand(owner.handle, ptr(pts), N, fx.sigma2, ptr(z), None, ptr(out), C.byref(il))
        else:
            rc = lib.lmm_imogp_rand(ctx.handle, _descs(f.fs), m, ptr(pts), N, D, fx.sigma2, p, ptr(z), ptr(out), C.byref(il))
        ctx.check(rc, il.value)
        if by_features:  # src/independent_mogp.jl:217-220
            return out.reshape(m, N).T.reshape(-1).copy()
        return out
    raise TypeError(f"rand not defined for FiniteGP of {type(f).__name__}")


def _terms_grads(fs, gt: np.ndarray, D: int) -> list:
    """grad_terms (m x LMM_MAX_TERMS x LMM_GRAD_TERM_STRIDE) -> per latent, one dict per term in Kernel.all_terms() order."""
    out = []
    for i, g in enumerate(fs):
        k = (g.prior if isinstance(g, PosteriorGP) else g).kernel
        rows = gt.reshape(len(fs), _lib.LMM_MAX_TERMS, _lib.LMM_GRAD_TERM_STRIDE)[i]
        out.append([{"variance": float(r[0]), "inv_lengthscale": float(r[1]), "param": float(r[2]), "ard": r[3:3 + D].copy()}
                    for r in rows[:len(k.all_terms())]])
    return out


def logpdf_and_gradient(fx: FiniteGP, y, with_grad_y: bool = False, kernel_terms: bool = False):
    """Value and gradient of `logpdf(fx, y)` for an OILMM, general ILMM or IndependentMOGP prior -- the pullback
    a ChainRulesCore `rrule` around the ccall returns (test/oilmm.jl:31-32, test/ilmm.jl:31 `gradient(logpdf, fx, y)`).
    A general ILMM returns "H" (p, m) instead of "U"/"S".
    Returns (logpdf, grads) with grads = {"variance": (m,), "inv_lengthscale": (m,), "mean_const": (m,),
    "sigma2": float[, "y": (p*N,)][, "U": (p, m), "S": (m,) for an OILMM]}.

    Composite (KernelSum / KernelProduct), PeriodicKernel and RationalQuadraticKernel latents need `kernel_terms=True`
    (without it a composite latent raises ValueError).  It adds grads["terms"]: per latent, a list in `Kernel.all_terms()`
    order of {"variance", "inv_lengthscale", "param" (α / r; 0 for kinds without one), "ard" (D,)} -- the gradient w.r.t.
    each term's own hyper-parameters; "variance" / "inv_lengthscale" / "ard" then hold term 0's.  A transform shared by all
    terms is a function of them: for `(k1 + k2) ∘ ScaleTransform(s)` each term carries s_t = s·c_t, so
    d/ds = Σ_t (s_t / s)·terms[t]["inv_lengthscale"].  On a posterior FiniteGP this gives σ² and y* only, with the
    posterior's data and hyper-parameters held fixed, and `kernel_terms=True` raises ValueError: the gradient through the
    conditioning is `predictive_logpdf_and_gradient`."""
    f = fx.f
    ctx = _ctx_of(fx)
    _require_by_outputs(fx)
    pts = _points(fx.x.x)
    N, D = int(pts.shape[0]), int(pts.shape[1])
    out, gs2, il = C.c_double(), C.c_double(), C.c_int(-1)
    yv = _yvec(y, N * fx.x.out_dim)
    gy = np.zeros(N * fx.x.out_dim) if with_grad_y else None
    owner = _post_owner(fx)
    if owner is not None:
        if kernel_terms:
            raise ValueError("kernel_terms: the posterior-predictive logpdf gradient covers σ² and y* only")
        # logpdf(post(x*, σ²), y*): gradient w.r.t. σ² and y* (test/oilmm.jl:32 `gradient(logpdf, po, y_test)`)
        if isinstance(f, ILMM) and f.H.shape[0] != fx.x.out_dim:
            raise RuntimeError("out dim of x != out dim of f.")
        rc = ctx.lib.lmm_post_logpdf_grad(owner.handle, ptr(pts), N, fx.sigma2, ptr(yv), C.byref(out), C.byref(gs2), ptr(gy), C.byref(il))
        ctx.check(rc, il.value)
        grads = {"sigma2": gs2.value}
        if with_grad_y:
            grads["y"] = gy
        return out.value, grads
    if isinstance(f, ILMM) and isinstance(f.H, Orthogonal) and isinstance(f.f, IndependentMOGP):
        lat, H = f.f, f.H
        m = len(lat.fs)
        gl = np.zeros((m, 3))
        gU = np.zeros(H.shape, order="F")
        gS = np.zeros(m)
        ga = np.zeros((m, D))
        fs = lat.fs
        args = (ctx.handle, _descs(fs), m, ptr(pts), N, D, ptr(H.U), ptr(H.S), H.shape[0], fx.sigma2, ptr(yv), fx.x.out_dim, C.byref(out),
                ptr(gl), ptr(ga), C.byref(gs2), ptr(gy), ptr(gU), ptr(gS))
        if kernel_terms:
            gt = np.zeros(m * _lib.LMM_MAX_TERMS * _lib.LMM_GRAD_TERM_STRIDE)
            rc = ctx.lib.lmm_oilmm_logpdf_grad_terms(*args, ptr(gt), C.byref(il))
        else:
            rc = ctx.lib.lmm_oilmm_logpdf_grad(*args, C.byref(il))
    elif isinstance(f, IndependentMOGP):
        m = len(f.fs)
        gl = np.zeros((m, 3))
        ga = np.zeros((m, D))
        fs = f.fs
        args = (ctx.handle, _descs(fs), m, ptr(pts), N, D, fx.sigma2, ptr(yv), fx.x.out_dim, C.byref(out), ptr(gl), ptr(ga), C.byref(gs2),
                ptr(gy))
        if kernel_terms:
            gt = np.zeros(m * _lib.LMM_MAX_TERMS * _lib.LMM_GRAD_TERM_STRIDE)
            rc = ctx.lib.lmm_imogp_logpdf_grad_terms(*args, ptr(gt), C.byref(il))
        else:
            rc = ctx.lib.lmm_imogp_logpdf_grad(*args, C.byref(il))
    elif isinstance(f, ILMM) and isinstance(f.f, IndependentMOGP):  # general mixing matrix, src/ilmm.jl:150-163
        lat = f.f
        m = len(lat.fs)
        Hm = as_f64(np.asarray(f.H), "F")
        gl = np.zeros((m, 3))
        gH = np.zeros(Hm.shape, order="F")
        ga = np.zeros((m, D))
        args = (ctx.handle, _descs(lat.fs), m, ptr(pts), N, D, ptr(Hm), Hm.shape[0], fx.sigma2, ptr(yv), fx.x.out_dim, C.byref(out), ptr(gl),
                ptr(ga), C.byref(gs2), ptr(gy), ptr(gH))
        if kernel_terms:
            gt = np.zeros(m * _lib.LMM_MAX_TERMS * _lib.LMM_GRAD_TERM_STRIDE)
            rc = ctx.lib.lmm_ilmm_logpdf_grad_terms(*args, ptr(gt), C.byref(il))
        else:
            rc = ctx.lib.lmm_ilmm_logpdf_grad(*args, C.byref(il))
        ctx.check(rc, il.value)
        grads = {"variance": gl[:, 0].copy(), "inv_lengthscale": gl[:, 1].copy(), "mean_const": gl[:, 2].copy(), "sigma2": gs2.value,
                 "H": np.ascontiguousarray(gH), "ard": ga}
        if kernel_terms:
            grads["terms"] = _terms_grads(lat.fs, gt, D)
        if with_grad_y:
            grads["y"] = gy
        return out.value, grads
    else:
        raise TypeError("logpdf_and_gradient is built for OILMM, ILMM and IndependentMOGP priors")
    ctx.check(rc, il.value)
    grads = {"variance": gl[:, 0].copy(), "inv_lengthscale": gl[:, 1].copy(), "mean_const": gl[:, 2].copy(), "sigma2": gs2.value,
             "ard": ga}  # (m, D): d/d ARDTransform multipliers, zeros for latents without one
    if kernel_terms:
        grads["terms"] = _terms_grads(fs, gt, D)
    if with_grad_y:
        grads["y"] = gy
    if isinstance(f, ILMM):
        grads["U"], grads["S"] = np.ascontiguousarray(gU), gS
    return out.value, grads


def predictive_logpdf_and_gradient(fx_post: FiniteGP, y, y_train, with_grad_y: bool = False):
    """Value and gradient of the posterior-predictive logpdf `logpdf(posterior(f(x, σ²), y_train)(x*, σ*²), y)`
    differentiated through the conditioning: the held-out / forecast likelihood, or the likelihood of new data given old,
    as a function of everything the posterior was built from.  `fx_post` is `post(x*, σ*²)` for a posterior of an OILMM
    or an IndependentMOGP (a masked OILMM posterior counts as an OILMM over its observed inputs); `y_train` is the data
    it was conditioned on (p*N by outputs; checked against the posterior).  Joint posteriors (general ILMM, dense Σy,
    missing data through the dense model) and posteriors conditioned a second time raise ValueError.

    Returns (logpdf, grads) with grads = {
      "sigma2": d/dσ*² (float)[, "y": d/dy* (p*Ns,)] -- exactly what `logpdf_and_gradient` returns on the posterior,
      "terms": per latent, per term in `Kernel.all_terms()` order, {"variance", "inv_lengthscale", "param", "ard" (D,)},
      "variance", "inv_lengthscale", "ard" (m, D): term 0's, "mean_const" (m,),
      "train": {"sigma2": d/dσ², "y": d/dy_train (p*N,)},
      "U" (p, m), "S" (m,) for an OILMM: the Euclidean gradient, as `logpdf_and_gradient` returns it}.
    Hyper-parameters enter the training and the test side through the same kernel, so each entry is the total derivative.
    A transform shared by all terms is a function of them: for `(k1 + k2) ∘ ScaleTransform(s)` each term carries
    s_t = s·c_t, so d/ds = Σ_t (s_t / s)·terms[t]["inv_lengthscale"]."""
    f = fx_post.f
    ctx = _ctx_of(fx_post)
    _require_by_outputs(fx_post)
    owner = _post_owner(fx_post)
    if owner is None:
        raise TypeError("predictive_logpdf_and_gradient needs a posterior FiniteGP, post(x*, σ²)")
    lat = f.f if isinstance(f, ILMM) else f
    if isinstance(f, ILMM) and f.H.shape[0] != fx_post.x.out_dim:
        raise RuntimeError("out dim of x != out dim of f.")
    pts = _points(fx_post.x.x)
    Ns, D = int(pts.shape[0]), int(pts.shape[1])
    p = fx_post.x.out_dim
    yv = _yvec(y, Ns * p)
    ytr = _yvec(y_train, owner.N * p)
    fs = lat.fs if isinstance(lat, IndependentMOGP) else lat.prior.fs if isinstance(lat, _JointPosterior) else []
    m = len(fs)
    orth = isinstance(f, ILMM) and isinstance(f.H, Orthogonal)
    out, gs2, gts2, il = C.c_double(), C.c_double(), C.c_double(), C.c_int(-1)
    gy = np.zeros(Ns * p) if with_grad_y else None
    gl = np.zeros((m, 3))
    ga = np.zeros((m, D))
    gt = np.zeros(m * _lib.LMM_MAX_TERMS * _lib.LMM_GRAD_TERM_STRIDE)
    gty = np.zeros(owner.N * p)
    gU = np.zeros((p, m), order="F") if orth else None
    gS = np.zeros(m) if orth else None
    rc = ctx.lib.lmm_post_logpdf_grad_full(owner.handle, ptr(pts), Ns, fx_post.sigma2, ptr(yv), ptr(ytr), C.byref(out), C.byref(gs2),
                                           ptr(gy), ptr(gl), ptr(ga), ptr(gt), C.byref(gts2), ptr(gty), ptr(gU), ptr(gS), C.byref(il))
    ctx.check(rc, il.value)
    grads = {"sigma2": gs2.value, "terms": _terms_grads(fs, gt, D), "variance": gl[:, 0].copy(), "inv_lengthscale": gl[:, 1].copy(),
             "ard": ga, "mean_const": gl[:, 2].copy(), "train": {"sigma2": gts2.value, "y": gty}}
    if with_grad_y:
        grads["y"] = gy
    if orth:
        grads["U"], grads["S"] = np.ascontiguousarray(gU), gS
    return out.value, grads


def _loo_call(fx: FiniteGP, y, value: bool, marginals: bool, grads: bool, with_grad_y: bool = False):
    """One lmm_oilmm_loo / lmm_imogp_loo call; outputs that are not asked for are passed as NULL."""
    if isinstance(fx.f, ILMM) and not isinstance(fx.f.H, Orthogonal):
        raise TypeError("leave-one-out is built for OILMM and IndependentMOGP priors (not a general ILMM)")
    if not (isinstance(fx.f, (ILMM, IndependentMOGP))):
        raise TypeError("leave-one-out is built for OILMM and IndependentMOGP priors")
    if fx.noise is not None:
        raise TypeError("leave-one-out needs scalar observation noise")
    _require_by_outputs(fx)
    if _post_owner(fx) is not None:
        raise TypeError("leave-one-out is built for prior FiniteGPs, not posteriors")
    f = fx.f
    lat = f.f if isinstance(f, ILMM) else f
    if not isinstance(lat, IndependentMOGP):
        raise TypeError("ILMM latents must be an IndependentMOGP")
    if isinstance(f, ILMM) and f.H.shape[0] != fx.x.out_dim:
        raise RuntimeError("out dim of x != out dim of f.")
    ctx = _ctx_of(fx)
    pts = _points(fx.x.x)
    N, D = int(pts.shape[0]), int(pts.shape[1])
    p = fx.x.out_dim
    m = len(lat.fs)
    yv = _yvec(y, N * p)
    if not _is_device_tensor(yv) and np.isnan(yv).any():
        raise ValueError("y has a NaN entry: leave-one-out needs fully observed data")
    out, gs2, il = C.c_double(), C.c_double(), C.c_int(-1)
    M = np.zeros(p * N) if marginals else None
    V = np.zeros(p * N) if marginals else None
    gl = np.zeros((m, 3)) if grads else None
    ga = np.zeros((m, D)) if grads else None
    gt = np.zeros(m * _lib.LMM_MAX_TERMS * _lib.LMM_GRAD_TERM_STRIDE) if grads else None
    gy = np.zeros(p * N) if grads and with_grad_y else None
    gs2p = C.byref(gs2) if grads else None
    outp = C.byref(out) if value else None
    orth = isinstance(f, ILMM)
    gU = np.zeros(f.H.shape, order="F") if orth and grads else None
    gS = np.zeros(m) if orth and grads else None
    if orth:
        H = f.H
        rc = ctx.lib.lmm_oilmm_loo(ctx.handle, _descs(lat.fs), m, ptr(pts), N, D, ptr(H.U), ptr(H.S), H.shape[0], fx.sigma2, ptr(yv), p,
                                   outp, ptr(M), ptr(V), ptr(gl), ptr(ga), gs2p, ptr(gy), ptr(gU), ptr(gS), ptr(gt), C.byref(il))
    else:
        rc = ctx.lib.lmm_imogp_loo(ctx.handle, _descs(lat.fs), m, ptr(pts), N, D, fx.sigma2, ptr(yv), p, outp, ptr(M), ptr(V), ptr(gl),
                                   ptr(ga), gs2p, ptr(gy), ptr(gt), C.byref(il))
    ctx.check(rc, il.value)
    g = None
    if grads:
        g = {"terms": _terms_grads(lat.fs, gt, D), "variance": gl[:, 0].copy(), "inv_lengthscale": gl[:, 1].copy(), "ard": ga,
             "mean_const": gl[:, 2].copy(), "sigma2": gs2.value}
        if with_grad_y:
            g["y"] = gy
        if orth:
            g["U"], g["S"] = np.ascontiguousarray(gU), gS
    return out.value, M, V, g


def loo_logpdf(fx: FiniteGP, y) -> float:
    """Leave-one-input-out log predictive density Σ_i log p(y_i | y_{-i}) of an OILMM or IndependentMOGP prior `fx`, where
    y_i is all outputs at input x_i (Rasmussen & Williams §5.4.2): a cross-validation score in closed form, for comparing
    models and as a training objective.  Costs one factorisation and one triangular inverse per latent."""
    return _loo_call(fx, y, True, False, False)[0]


def loo_mean_and_var(fx: FiniteGP, y) -> Tuple[np.ndarray, np.ndarray]:
    """LOO predictive marginals (p*N each, by outputs like `mean_and_var`): at each input x_i, what
    `mean_and_var(posterior(f(x_{-i}, σ²), y_{-i})(x_i, σ²))` returns -- noise included."""
    _, M, V, _ = _loo_call(fx, y, False, True, False)
    return M, V


def loo_logpdf_and_gradient(fx: FiniteGP, y, with_grad_y: bool = False):
    """Value and gradient of `loo_logpdf(fx, y)`.  grads has the keys of `logpdf_and_gradient(fx, y, kernel_terms=True)`:
    "terms" (per latent, per term in `Kernel.all_terms()` order: {"variance", "inv_lengthscale", "param", "ard"}),
    "variance" / "inv_lengthscale" / "ard" (term 0's), "mean_const", "sigma2"[, "y" (p*N,)], and for an OILMM "U" (p, m)
    and "S" (m,), the Euclidean gradient.  General ILMMs, posteriors, by-features inputs and non-scalar noise raise
    TypeError; a NaN in y raises ValueError."""
    v, _, _, g = _loo_call(fx, y, True, False, True, with_grad_y)
    return v, g


def logpdf_sweep(fx: FiniteGP, y, inv_lengthscale_scales) -> np.ndarray:
    """BASELINE config 5: OILMM logpdf for a batch of lengthscale settings in one call."""
    lat, H, s2, _ = unpack(fx)
    if not isinstance(H, Orthogonal):
        raise TypeError("logpdf_sweep needs an OILMM")
    ctx = _ctx_of(fx)
    pts = _points(fx.x.x)
    N, D = int(pts.shape[0]), int(pts.shape[1])
    m = len(lat.fs)
    sc = as_f64(inv_lengthscale_scales).reshape(-1)
    out = np.zeros(sc.shape[0])
    il = C.c_int(-1)
    yv = _yvec(y, N * fx.x.out_dim)
    rc = ctx.lib.lmm_oilmm_logpdf_sweep(ctx.handle, _descs(lat.fs), m, ptr(pts), N, D, ptr(H.U), ptr(H.S), H.shape[0], s2, ptr(yv),
                                        fx.x.out_dim, ptr(sc), sc.shape[0], ptr(out), C.byref(il))
    ctx.check(rc, il.value)
    return out


def potrf_batched(A: np.ndarray, ctx: Optional[Context] = None):
    """Batched blocked Cholesky of `A[b]` (symmetric, lower read): returns (L, logdet, info)."""
    ctx = ctx or default_context()
    A = np.asarray(A, dtype=np.float64)
    if A.ndim == 2:
        A = A[None]
    batch, N, _ = A.shape
    Af = np.ascontiguousarray(np.transpose(A, (0, 2, 1)))  # each matrix column-major
    L = np.zeros_like(Af)
    logdet = np.zeros(batch)
    info = np.zeros(batch, dtype=np.int32)
    rc = ctx.lib.lmm_potrf_batched(ctx.handle, ptr(Af), N, batch, ptr(L), ptr(logdet), ptr(info))
    if rc < 0:
        ctx.check(rc)
    return np.transpose(L, (0, 2, 1)), logdet, info


def save_posterior(post, path: str) -> None:
    """Write a posterior (as returned by `posterior`) to `path`: metadata + device arrays verbatim (lmm_post_save)."""
    owner = _post_owner(FiniteGP(post, MOInputIsotopicByOutputs(np.zeros(1), 1)))
    if owner is None:
        raise TypeError("save_posterior needs a posterior returned by `posterior`")
    owner.ctx.check(owner.ctx.lib.lmm_post_save(owner.handle, os.fsencode(path)))


def load_posterior(path: str, prior, ctx: Optional[Context] = None):
    """Restore a posterior saved by `save_posterior`.  `prior` is the model it was conditioned from (ILMM / OILMM /
    IndependentMOGP): it supplies the host-side wrappers, every number comes from the file."""
    ctx = ctx or default_context()
    h = C.c_void_p()
    ctx.check(ctx.lib.lmm_post_load(ctx.handle, os.fsencode(path), C.byref(h)))
    kind, m, p, N, D = C.c_int(), C.c_int(), C.c_int(), C.c_int(), C.c_int()
    nbytes = C.c_int64()
    ctx.check(ctx.lib.lmm_post_info(h, C.byref(kind), C.byref(m), C.byref(p), C.byref(N), C.byref(D), C.byref(nbytes)))
    lat = prior.f if isinstance(prior, ILMM) else prior
    if isinstance(lat, _JointPosterior):
        lat = lat.prior
    priors = [g.prior if isinstance(g, PosteriorGP) else g for g in lat.fs]
    if len(priors) != m.value:
        ctx.lib.lmm_post_free(h)
        raise ValueError("the prior model does not match the saved posterior")
    if kind.value == 4:  # missing-data posterior of the dense model
        return _MissingDataPosterior(_PostHandle(ctx, h, N.value), prior, 0)
    if kind.value in (2, 3):  # joint factor: general ILMM / IndependentMOGP under a dense Σy
        joint = _JointPosterior(_PostHandle(ctx, h, N.value, joint_n=m.value * N.value), IndependentMOGP(priors))
        return ILMM(joint, prior.H) if kind.value == 2 else joint
    owner = _PostHandle(ctx, h, N.value)
    newlat = IndependentMOGP([PosteriorGP(owner, i, g) for i, g in enumerate(priors)])
    return ILMM(newlat, prior.H) if kind.value == 0 else newlat


class _MissingDataPosterior(AbstractGP):
    """Posterior of an ILMM / OILMM conditioned on a partially observed y (NaN = missing) through the dense multi-output model:
    `mean_and_var` / `mean` / `var` / `marginals` / `mean_and_cov` / `cov` / `rand` at new inputs for all outputs, save / load."""

    def __init__(self, owner: _PostHandle, prior: ILMM, n_observed: int):
        self._owner, self.prior, self.n_observed = owner, prior, n_observed


def _nan_mask_is_per_input(y: np.ndarray, p: int, N: int) -> bool:
    nan = np.isnan(y.reshape(p, N))
    cnt = nan.sum(axis=0)
    return bool(np.all((cnt == 0) | (cnt == p)))


def posterior_missing(fx: FiniteGP, y, with_logpdf: bool = False):
    """Heterotopic / missing-data conditioning (SURVEY §8f-4; the reference leaves it unsupported): entries of `y` that are NaN
    are unobserved.  An OILMM whose mask is per input (whole time steps missing) stays an OILMM on the observed inputs --
    per-latent O(m N_obs³), and the result is an ordinary OILMM posterior with every method; any other mask is conditioned
    exactly on the observed entries of the dense multi-output model (`ILMM(fs, H)` with a dense or an `Orthogonal` H) and
    returns a posterior whose FiniteGPs answer `mean_and_var` / `mean` / `var` / `marginals` / `mean_and_cov` / `cov` / `rand`."""
    lat, H, s2, _ = unpack(fx)
    if not isinstance(lat, IndependentMOGP) or any(isinstance(g, PosteriorGP) for g in lat.fs):
        raise TypeError("posterior_missing needs an ILMM / OILMM over prior latents")
    ctx = default_context()
    pts = _points(fx.x.x)
    N, D = int(pts.shape[0]), int(pts.shape[1])
    Hm = as_f64(np.asarray(H), "F")
    p, m = Hm.shape
    yv = np.ascontiguousarray(np.asarray(y, dtype=np.float64).reshape(-1))
    if yv.shape[0] != N * p:
        raise ValueError("length of y does not match the inputs")
    h, out, nobs, info = C.c_void_p(), C.c_double(), C.c_int(0), C.c_int(0)
    if isinstance(H, Orthogonal) and _nan_mask_is_per_input(yv, p, N):
        rc = ctx.lib.lmm_oilmm_masked_posterior(ctx.handle, _descs(lat.fs), m, ptr(pts), N, D, ptr(H.U), ptr(H.S), p, s2, ptr(yv), fx.x.out_dim,
                                                C.byref(h), C.byref(out), C.byref(nobs), C.byref(info))
        ctx.check(rc, info.value)
        owner = _PostHandle(ctx, h, nobs.value)
        post = ILMM(IndependentMOGP([PosteriorGP(owner, i, g) for i, g in enumerate(lat.fs)]), H)
        return (post, out.value) if with_logpdf else post
    rc = ctx.lib.lmm_ilmm_masked_posterior(ctx.handle, _descs(lat.fs), m, ptr(pts), N, D, ptr(Hm), p, s2, ptr(yv), fx.x.out_dim, C.byref(h),
                                           C.byref(out), C.byref(nobs), C.byref(info))
    ctx.check(rc)
    post = _MissingDataPosterior(_PostHandle(ctx, h, N, joint_n=nobs.value), fx.f, nobs.value)
    return (post, out.value) if with_logpdf else post


def logpdf_missing(fx: FiniteGP, y) -> float:
    """logpdf of the observed (non-NaN) entries of `y` under the ILMM / OILMM `fx` (per-input masks of an OILMM: the OILMM
    logpdf on the observed inputs; otherwise the dense model)."""
    lat, H, s2, _ = unpack(fx)
    ctx = default_context()
    pts = _points(fx.x.x)
    N, D = int(pts.shape[0]), int(pts.shape[1])
    Hm = as_f64(np.asarray(H), "F")
    p, m = Hm.shape
    yv = np.ascontiguousarray(np.asarray(y, dtype=np.float64).reshape(-1))
    out, info = C.c_double(), C.c_int(0)
    if isinstance(H, Orthogonal) and _nan_mask_is_per_input(yv, p, N):
        rc = ctx.lib.lmm_oilmm_masked_posterior(ctx.handle, _descs(lat.fs), m, ptr(pts), N, D, ptr(H.U), ptr(H.S), p, s2, ptr(yv), fx.x.out_dim,
                                                None, C.byref(out), None, C.byref(info))
        ctx.check(rc, info.value)
        return out.value
    rc = ctx.lib.lmm_ilmm_masked_posterior(ctx.handle, _descs(lat.fs), m, ptr(pts), N, D, ptr(Hm), p, s2, ptr(yv), fx.x.out_dim, None,
                                           C.byref(out), None, C.byref(info))
    ctx.check(rc)
    return out.value


def logpdf_missing_and_gradient(fx: FiniteGP, y, with_grad_y: bool = False, kernel_terms: bool = False):
    """Value and gradient of `logpdf_missing(fx, y)`: entries of `y` that are NaN are unobserved.  Routes as
    `logpdf_missing` does.  An OILMM (`Orthogonal` H) with a per-input mask is the OILMM gradient on the observed inputs and
    returns "U" / "S" as `logpdf_and_gradient` does.  Any other model or mask runs the dense model on the observed entries
    and returns "H" (p, m), d/dH of C_ab = Σ_l H[j_a,l] H[j_b,l] k_l + σ²[a = b].  With an `Orthogonal` H it also returns
    "U" = gH·diag(√S) and "S"[l] = Σ_j gH[j,l] U[j,l] / (2√S_l), the chain rule of H = U√S.  That is the Euclidean
    gradient of the dense-model expression: it agrees with the OILMM path's "U" in the tangent space of orthogonal U
    (after projecting G -> G - U sym(U'G)), not off it.
    "variance" / "inv_lengthscale" / "mean_const" / "sigma2" / "ard" / "terms" mean what they mean in
    `logpdf_and_gradient` (composite latents need `kernel_terms=True`); "y" (p*N,) is 0 at every NaN entry.  A posterior
    FiniteGP raises TypeError."""
    lat, H, s2, _ = unpack(fx)
    if not isinstance(lat, IndependentMOGP) or any(isinstance(g, PosteriorGP) for g in lat.fs):
        raise TypeError("logpdf_missing_and_gradient needs an ILMM / OILMM over prior latents")
    ctx = default_context()
    pts = _points(fx.x.x)
    N, D = int(pts.shape[0]), int(pts.shape[1])
    Hm = as_f64(np.asarray(H), "F")
    p, m = Hm.shape
    yv = np.ascontiguousarray(np.asarray(y, dtype=np.float64).reshape(-1))
    if yv.shape[0] != N * p:
        raise ValueError("length of y does not match the inputs")
    out, gs2, nobs, info = C.c_double(), C.c_double(), C.c_int(0), C.c_int(-1)
    gl = np.zeros((m, 3))
    ga = np.zeros((m, D))
    gy = np.zeros(N * p) if with_grad_y else None
    gt = np.zeros(m * _lib.LMM_MAX_TERMS * _lib.LMM_GRAD_TERM_STRIDE) if kernel_terms else None
    if isinstance(H, Orthogonal) and _nan_mask_is_per_input(yv, p, N):
        gU = np.zeros(H.shape, order="F")
        gS = np.zeros(m)
        rc = ctx.lib.lmm_oilmm_masked_logpdf_grad(ctx.handle, _descs(lat.fs), m, ptr(pts), N, D, ptr(H.U), ptr(H.S), p, s2, ptr(yv),
                                                  fx.x.out_dim, C.byref(out), ptr(gl), ptr(ga), C.byref(gs2), ptr(gy), ptr(gU), ptr(gS),
                                                  ptr(gt), C.byref(nobs), C.byref(info))
        ctx.check(rc, info.value)
        grads = {"U": np.ascontiguousarray(gU), "S": gS}
    else:
        gH = np.zeros((p, m), order="F")
        rc = ctx.lib.lmm_ilmm_masked_logpdf_grad(ctx.handle, _descs(lat.fs), m, ptr(pts), N, D, ptr(Hm), p, s2, ptr(yv), fx.x.out_dim,
                                                 C.byref(out), ptr(gl), ptr(ga), C.byref(gs2), ptr(gy), ptr(gH), ptr(gt), C.byref(nobs),
                                                 C.byref(info))
        ctx.check(rc)
        grads = {"H": np.ascontiguousarray(gH)}
        if isinstance(H, Orthogonal):
            rs = np.sqrt(np.asarray(H.S, dtype=np.float64))
            grads["U"] = grads["H"] * rs[None, :]
            grads["S"] = np.sum(grads["H"] * np.asarray(H.U), axis=0) / (2.0 * rs)
    grads.update({"variance": gl[:, 0].copy(), "inv_lengthscale": gl[:, 1].copy(), "mean_const": gl[:, 2].copy(), "sigma2": gs2.value,
                  "ard": ga})
    if kernel_terms:
        grads["terms"] = _terms_grads(lat.fs, gt, D)
    if with_grad_y:
        grads["y"] = gy
    return out.value, grads
