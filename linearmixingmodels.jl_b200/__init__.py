"""B200-native (sm_100a) inference hot path of LinearMixingModels.jl.

The directory name carries a dot, so import it through the root-level alias module:

    import lmm_b200 as lmm

Only what the path needs lives here: `csrc/` (CUDA kernels + the C ABI -> liblmm.so), the ctypes
binding (`_lib.py`), the host-side mirror of the reference interface (`api.py`), the multi-GPU
plumbing (`dist.py`) and the Julia shim source (`julia/`).
"""
from .api import *  # noqa: F401,F403
from .api import (  # noqa: F401
    logpdf_terms,
    logpdf_sweep,
    logpdf_and_gradient,
    predictive_logpdf_and_gradient,
    potrf_batched,
    set_default_context,
    set_ilmm_form,
    save_posterior,
    load_posterior,
    posterior_missing,
    logpdf_missing,
    logpdf_missing_and_gradient,
    loo_logpdf,
    loo_mean_and_var,
    loo_logpdf_and_gradient,
)
from . import _lib, api, dist  # noqa: F401

__version__ = "0.1.0"
