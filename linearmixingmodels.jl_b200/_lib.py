"""ctypes binding of liblmm.so (include/lmm.h).  No fallback: a missing library or a missing
CUDA device is a hard error -- the product path never routes through the CPU oracle."""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblmm.so")

LMM_OK = 0
LMM_E_ARG, LMM_E_OUT_DIM, LMM_E_UNSUPPORTED, LMM_E_CUDA, LMM_E_NCCL, LMM_E_NOT_ORTHOGONAL, LMM_E_OOM = -1, -2, -3, -4, -5, -6, -7
LMM_MAX_TERMS, LMM_MAX_ARD = 4, 8
LMM_GRAD_TERM_STRIDE = 3 + LMM_MAX_ARD  # per term: d/d variance, d/d inv_lengthscale, d/d param, d/d ard[0..8)


class LibraryNotBuilt(ImportError):
    pass


class PosDefException(np.linalg.LinAlgError):
    """Mirror of Julia's PosDefException(info) raised by a failed `cholesky`."""

    def __init__(self, info: int, latent: int = -1, msg: str = ""):
        super().__init__(msg or f"matrix is not positive definite; Cholesky factorization failed (info={info}, latent={latent})")
        self.info = info
        self.latent = latent


class KernelTerm(C.Structure):  # lmm_kernel_term: one further term of a composite (sum / product) kernel
    _fields_ = [
        ("kind", C.c_int32),
        ("reserved", C.c_int32),
        ("variance", C.c_double),
        ("inv_lengthscale", C.c_double),
        ("param", C.c_double),
        ("ard", C.c_void_p),
    ]


class GpDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("compose", C.c_int32),  # 0 single kernel, 1 KernelSum, 2 KernelProduct over this term and `extra`
        ("variance", C.c_double),
        ("inv_lengthscale", C.c_double),
        ("mean_const", C.c_double),
        ("ard", C.c_void_p),  # const double*: D per-dimension multipliers (ARDTransform) or NULL
        ("param", C.c_double),  # α of RationalQuadraticKernel, r of PeriodicKernel
        ("n_extra", C.c_int32),
        ("reserved2", C.c_int32),
        ("extra", C.c_void_p),  # const lmm_kernel_term*: n_extra further terms or NULL
    ]

    def __init__(self, kind=0, compose=0, variance=1.0, inv_lengthscale=1.0, mean_const=0.0, ard=None, param=1.0, n_extra=0, reserved2=0, extra=None):
        super().__init__(kind, compose, variance, inv_lengthscale, mean_const, ard, param, n_extra, reserved2, extra)


_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_vp = C.c_void_p

# name -> (restype, argtypes); every symbol include/lmm.h declares.
SIGNATURES = {
    "lmm_ctx_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "lmm_ctx_destroy": (C.c_int, [_vp]),
    "lmm_last_error": (C.c_char_p, [_vp]),
    "lmm_version": (C.c_char_p, []),
    "lmm_ctx_set_option": (C.c_int, [_vp, C.c_char_p, C.c_double]),
    "lmm_ctx_counters": (C.c_int, [_vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "lmm_ctx_last_timings": (C.c_int, [_vp, _dp]),
    "lmm_comm_unique_id": (C.c_int, [_vp]),
    "lmm_comm_init": (C.c_int, [_vp, _vp, C.c_int, C.c_int]),
    "lmm_comm_set_shard": (C.c_int, [_vp, C.c_int, C.c_int]),
    "lmm_orthogonal_validate": (C.c_int, [_vp, C.c_int, C.c_int]),
    "lmm_oilmm_logpdf": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, C.c_int, _dp, _vp, _ip]),
    "lmm_oilmm_posterior": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, C.c_int, C.POINTER(_vp), _dp, _vp, _ip]),
    "lmm_oilmm_prior_mean_and_var": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, C.c_int, _vp, _vp]),
    "lmm_oilmm_rand": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, C.c_int, _vp, _vp, _vp, _ip]),
    "lmm_oilmm_logpdf_sweep": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, C.c_int, _vp, C.c_int, _vp, _ip]),
    "lmm_oilmm_logpdf_grad": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, C.c_int, _dp, _vp, _vp, _dp, _vp, _vp, _vp, _ip]),
    "lmm_imogp_logpdf_grad": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, C.c_double, _vp, C.c_int, _dp, _vp, _vp, _dp, _vp, _ip]),
    # per-term gradients of composite / periodic / rational-quadratic latents: grad_terms (m x 4 x 11) before the info pointer
    "lmm_oilmm_logpdf_grad_terms": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, C.c_int, _dp, _vp, _vp, _dp, _vp, _vp, _vp, _vp, _ip]),
    "lmm_imogp_logpdf_grad_terms": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, C.c_double, _vp, C.c_int, _dp, _vp, _vp, _dp, _vp, _vp, _ip]),
    # leave-one-input-out: value, LOO mean, LOO var, latents, ard, σ², y, U, S, terms, info
    "lmm_oilmm_loo": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, C.c_int, _dp, _vp, _vp, _vp, _vp, _dp, _vp, _vp, _vp, _vp, _ip]),
    "lmm_imogp_loo": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, C.c_double, _vp, C.c_int, _dp, _vp, _vp, _vp, _vp, _dp, _vp, _vp, _ip]),
    "lmm_post_mean_and_var": (C.c_int, [_vp, _vp, C.c_int, C.c_double, _vp, _vp]),
    "lmm_post_latent_mean_and_var": (C.c_int, [_vp, C.c_int, _vp, C.c_int, C.c_double, _vp, _vp]),
    "lmm_post_mean_and_cov": (C.c_int, [_vp, _vp, C.c_int, C.c_double, _vp, _vp]),
    "lmm_prior_mean_and_cov": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, C.c_int, C.c_double, C.c_double, C.c_int, _vp, _vp]),
    "lmm_post_condition": (C.c_int, [_vp, _vp, C.c_int, C.c_double, _vp, C.POINTER(_vp), _ip]),
    "lmm_post_logpdf": (C.c_int, [_vp, _vp, C.c_int, C.c_double, _vp, _dp, _ip]),
    "lmm_post_logpdf_grad": (C.c_int, [_vp, _vp, C.c_int, C.c_double, _vp, _dp, _dp, _vp, _ip]),
    # through the conditioning: y_train, value, σ*², y*, latents, ard, terms, training σ², training y, U, S, info
    "lmm_post_logpdf_grad_full": (C.c_int, [_vp, _vp, C.c_int, C.c_double, _vp, _vp, _dp, _dp, _vp, _vp, _vp, _vp, _dp, _vp, _vp, _vp, _ip]),
    "lmm_post_rand": (C.c_int, [_vp, _vp, C.c_int, C.c_double, _vp, _vp, _vp, _ip]),
    "lmm_post_export": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp]),
    "lmm_post_info": (C.c_int, [_vp, _ip, _ip, _ip, _ip, _ip, C.POINTER(C.c_int64)]),
    "lmm_post_save": (C.c_int, [_vp, C.c_char_p]),
    "lmm_post_load": (C.c_int, [_vp, C.c_char_p, C.POINTER(_vp)]),
    "lmm_post_free": (C.c_int, [_vp]),
    "lmm_imogp_logpdf": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, C.c_double, _vp, C.c_int, _dp, _vp, _ip]),
    "lmm_imogp_posterior": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, C.c_double, _vp, C.c_int, C.POINTER(_vp), _dp, _ip]),
    "lmm_imogp_posterior_noise": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, C.c_int, _vp, C.c_int, C.POINTER(_vp), _dp, _ip]),
    "lmm_imogp_rand": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, C.c_double, C.c_int, _vp, _vp, _ip]),
    "lmm_imogp_cross_cov": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp]),
    "lmm_reorder_indices": (C.c_int, [C.c_int, C.c_int, C.c_int, _vp]),
    "lmm_ilmm_logpdf": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, C.c_int, C.c_double, _vp, C.c_int, C.c_int, _dp, _ip]),
    "lmm_ilmm_posterior": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, C.c_int, C.c_double, _vp, C.c_int, C.POINTER(_vp), _dp, _ip]),
    "lmm_ilmm_prior_mean_and_var": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, C.c_int, C.c_double, C.c_int, _vp, _vp]),
    "lmm_ilmm_rand": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, C.c_int, C.c_double, C.c_int, _vp, _vp, _vp, _ip]),
    "lmm_ilmm_logpdf_grad": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, C.c_int, C.c_double, _vp, C.c_int, _dp, _vp, _vp, _dp, _vp, _vp, _ip]),
    "lmm_ilmm_logpdf_grad_terms": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, C.c_int, C.c_double, _vp, C.c_int, _dp, _vp, _vp, _dp, _vp, _vp, _vp, _ip]),
    "lmm_ilmm_masked_posterior": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, C.c_int, C.c_double, _vp, C.c_int, C.POINTER(_vp), _dp, _ip, _ip]),
    "lmm_oilmm_masked_posterior": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, C.c_int, C.POINTER(_vp), _dp, _ip, _ip]),
    # missing-data logpdf gradient: dense model (grad_terms nullable, n_observed, info) and per-input-mask OILMM
    "lmm_ilmm_masked_logpdf_grad": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, C.c_int, C.c_double, _vp, C.c_int, _dp, _vp, _vp, _dp, _vp, _vp, _vp, _ip, _ip]),
    "lmm_oilmm_masked_logpdf_grad": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_double, _vp, C.c_int, _dp, _vp, _vp, _dp, _vp, _vp, _vp, _vp, _ip, _ip]),
    "lmm_potrf_batched": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp, _vp, _vp]),
    "lmm_mvn_logpdf_rand": (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _dp, _vp, _vp, _ip]),
    "lmm_potrf_bench": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_double, C.c_int, _vp, _dp, _dp]),
}

_lib = None
_lock = threading.Lock()


def load():
    """Load liblmm.so and bind every declared symbol.  Raises LibraryNotBuilt if absent."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise LibraryNotBuilt(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  There is no CPU fallback."
            )
        lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def as_f64(a, order="C"):
    return np.require(np.asarray(a, dtype=np.float64), requirements=["A", order[0]])


def ptr(a):
    """Pointer to a NumPy array, a torch CUDA/CPU float64 tensor, or None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    raise TypeError(f"cannot take a pointer of {type(a)}")
