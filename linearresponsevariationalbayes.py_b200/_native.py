"""ctypes binding of liblrvb_b200.so (the C ABI declared in include/lrvb_b200.h).

There is no CPU fallback: if the shared library is missing or a CUDA device is absent, every
compute entry point raises.  PyTorch is used only as the device-memory container: tensors are
passed as raw ``data_ptr()`` addresses and all work is enqueued on torch's current stream.
"""
import ctypes
import os
from ctypes import POINTER, byref, c_char_p, c_double, c_int32, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# LRVB_LIB_PATH: another build of the same library (A/B timing of kernel changes)
LIB_PATH = os.environ.get("LRVB_LIB_PATH") or os.path.join(_HERE, "lib", "liblrvb_b200.so")

LRVB_OK, LRVB_EINVAL, LRVB_ECUDA, LRVB_ESTATE = 0, -1, -2, -3


class Prior(ctypes.Structure):
    """lrvb_glmm_prior (ExponentialFamilies.py:191-195 uvn_prior / gamma_prior arguments)."""
    _fields_ = [(n, c_double) for n in
                ("mu_mean", "mu_info", "beta_mean", "beta_info", "tau_shape", "tau_rate")]


class Bounds(ctypes.Structure):
    """lrvb_glmm_bounds (NormalParams.py:29,56 min_info; GammaParams.py:7-8 min_shape/min_rate)."""
    _fields_ = [(n, c_double) for n in ("mu_info", "tau_shape", "tau_rate", "beta_info", "u_info")]


class CGPrecond(ctypes.Structure):
    """lrvb_cg_precond: the `M=` of scipy.sparse.linalg.cg (ConjugateGradient.py:84) for the device CG."""
    _fields_ = [("kind", c_int32), ("Sinv_dev", c_void_p), ("indptr_dev", c_void_p),
                ("indices_dev", c_void_p), ("data_dev", c_void_p), ("dense_dev", c_void_p)]


PRECOND_NONE, PRECOND_BLOCK_JACOBI, PRECOND_SCHUR, PRECOND_CSR, PRECOND_DENSE = 0, 1, 2, 3, 4

# name -> (restype, argtypes); must list every symbol of include/lrvb_b200.h
_P = c_void_p
SIGNATURES = {
    "lrvb_last_error": (c_char_p, []),
    "lrvb_version": (c_int32, []),
    "lrvb_glmm_create": (c_int32, [POINTER(c_void_p), c_int64, c_int32, c_int32, c_int32, _P, _P,
                                   _P, _P, POINTER(c_double), POINTER(c_double), POINTER(Prior),
                                   POINTER(Bounds), c_int32, _P]),
    "lrvb_glmm_destroy": (c_int32, [_P]),
    "lrvb_launch_count": (ctypes.c_longlong, []),
    "lrvb_glmm_set_timing": (c_int32, [_P, c_int32]),
    "lrvb_glmm_last_timing": (c_int32, [_P, POINTER(ctypes.c_float)]),
    "lrvb_glmm_set_coords": (c_int32, [_P, c_int32]),
    "lrvb_glmm_set_shard": (c_int32, [_P, c_int64, c_int64]),
    "lrvb_glmm_dims": (c_int32, [_P, POINTER(c_int64), POINTER(c_int32)]),
    "lrvb_glmm_eval": (c_int32, [_P, _P, c_int32, _P, _P, _P]),
    "lrvb_glmm_blocks": (c_int32, [_P, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p)]),
    "lrvb_glmm_set_global_block": (c_int32, [_P, _P, _P]),
    "lrvb_glmm_result_buffers": (c_int32, [_P, POINTER(c_void_p), POINTER(c_void_p)]),
    "lrvb_glmm_obs_weights": (c_int32, [_P, POINTER(c_void_p), POINTER(c_int64)]),
    "lrvb_glmm_weight_cross_matvec": (c_int32, [_P, _P, _P, _P]),
    "lrvb_glmm_weight_cross_rmatvec": (c_int32, [_P, _P, _P, _P]),
    "lrvb_glmm_hessian_csr_capacity": (c_int32, [_P, POINTER(c_int64)]),
    "lrvb_glmm_hessian_csr": (c_int32, [_P, _P, _P, _P, c_int64, _P, _P]),
    "lrvb_glmm_hessian_csr_refill": (c_int32, [_P, _P, _P, _P, _P, _P]),
    "lrvb_glmm_hessian_csr_if": (c_int32, [_P, _P, _P, _P, _P, c_int64, _P, _P]),
    "lrvb_glmm_hvp": (c_int32, [_P, _P, _P, c_int32, _P]),
    "lrvb_glmm_cg": (c_int32, [_P, _P, _P, c_int32, c_double, c_int32, _P, POINTER(c_int32),
                               POINTER(c_int32), _P]),
    "lrvb_glmm_cg_m": (c_int32, [_P, _P, _P, POINTER(CGPrecond), c_double, c_int32, _P, POINTER(c_int32),
                                 POINTER(c_int32), _P]),
    "lrvb_glmm_schur": (c_int32, [_P, _P, c_int32, _P]),
    "lrvb_spd_inverse": (c_int32, [_P, c_int32, POINTER(c_int32), _P]),
    "lrvb_glmm_solve_reduce_rhs": (c_int32, [_P, _P, c_int32, _P, c_int32, _P]),
    "lrvb_glmm_solve_finish": (c_int32, [_P, _P, _P, _P, c_int32, _P, _P]),
    "lrvb_glmm_local_cov": (c_int32, [_P, _P, _P, _P]),
    "lrvb_glmm_predict": (c_int32, [_P, _P, _P, c_int32, _P, _P, c_int64, _P, _P]),
    "lrvb_glmm_predict_cross": (c_int32, [_P, _P, _P, _P]),
    "lrvb_glmm_predict_lr": (c_int32, [_P, _P, _P, _P, _P, c_int32, _P, _P, c_int64, _P, _P]),
    "lrvb_glmm_loo": (c_int32, [_P, _P, _P, _P, _P, _P]),
    "lrvb_glmm_logo": (c_int32, [_P, _P, _P, _P, _P, _P, _P]),
    "lrvb_glmm_third_contract": (c_int32, [_P, _P, _P, _P, _P]),
    "lrvb_ef_gamma_entropy": (c_int32, [_P, _P, c_int64, _P, _P]),
    "lrvb_ef_e_log_gamma": (c_int32, [_P, _P, c_int64, _P, _P]),
    "lrvb_ef_gamma_terms": (c_int32, [_P, _P, c_int64, _P, _P, _P]),
    "lrvb_ef_dirichlet_terms": (c_int32, [_P, c_int32, c_int64, _P, _P, _P]),
    "lrvb_ef_uvn_entropy": (c_int32, [_P, c_int64, _P, _P]),
    "lrvb_ef_dirichlet_entropy": (c_int32, [_P, c_int32, c_int64, _P, _P]),
    "lrvb_ef_e_log_dirichlet": (c_int32, [_P, c_int32, c_int64, _P, _P]),
    "lrvb_ef_beta_entropy": (c_int32, [_P, c_int64, _P, _P]),
    "lrvb_ef_wishart": (c_int32, [_P, _P, c_int32, c_int64, _P, _P, _P, _P]),
    "lrvb_ef_multinoulli_entropy": (c_int32, [_P, c_int32, c_int64, c_double, _P, _P]),
    "lrvb_gh_logistic_term": (c_int32, [_P, _P, c_int64, POINTER(c_double), POINTER(c_double),
                                        c_int32, _P, _P]),
    "lrvb_sum": (c_int32, [_P, c_int64, _P, _P]),
    "lrvb_posdef_unpack": (c_int32, [_P, c_int32, c_int64, c_double, _P, _P]),
    "lrvb_posdef_pack": (c_int32, [_P, c_int32, c_int64, c_double, _P, _P, _P]),
    "lrvb_posdef_free_to_vector": (c_int32, [_P, c_int32, c_int64, c_double, _P, _P]),
    "lrvb_posdef_free_to_vector_jac": (c_int32, [_P, c_int32, c_int64, c_double, _P, _P]),
    "lrvb_posdef_free_to_vector_hess": (c_int32, [_P, c_int32, c_int64, c_double, _P, _P]),
    "lrvb_simplex_constrain": (c_int32, [_P, c_int64, c_int32, _P, _P]),
    "lrvb_simplex_unconstrain": (c_int32, [_P, c_int64, c_int32, _P, _P]),
    "lrvb_simplex_jac": (c_int32, [_P, c_int64, c_int32, _P, _P]),
    "lrvb_simplex_hess": (c_int32, [_P, c_int64, c_int32, _P, _P]),
    "lrvb_p2p_create": (c_int32, [POINTER(c_void_p), c_int32, c_int32, c_int64]),
    "lrvb_p2p_handle_bytes": (c_int32, []),
    "lrvb_p2p_export": (c_int32, [_P, _P]),
    "lrvb_p2p_connect": (c_int32, [_P, _P]),
    "lrvb_p2p_allreduce_sum": (c_int32, [_P, _P, c_int64, _P]),
    "lrvb_p2p_status": (c_int32, [_P, POINTER(c_int32), _P]),
    "lrvb_p2p_status_nowait": (c_int32, [_P, POINTER(c_int32)]),
    "lrvb_p2p_set_timeout": (c_int32, [_P, c_double]),
    "lrvb_p2p_set_stats": (c_int32, [_P, c_int32, _P]),
    "lrvb_p2p_get_stats": (c_int32, [_P, POINTER(c_double), _P]),
    "lrvb_p2p_destroy": (c_int32, [_P]),
    "lrvb_glmm_cg_sharded": (c_int32, [_P, _P, _P, _P, c_int32, c_double, c_int32, c_int32, _P,
                                       POINTER(c_int32), POINTER(c_int32), _P]),
}

_lib = None


def load():
    """Loads the shared library (once).  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "lrvb_b200: %s is missing. Build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (needs nvcc). There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    msg = load().lrvb_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc):
    """Maps C status codes to the reference's exception types (SURVEY.md 8b)."""
    if rc == LRVB_OK:
        return
    msg = last_error()
    if rc == LRVB_EINVAL:
        raise ValueError(msg)
    raise RuntimeError(msg)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("lrvb_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return c_void_p(0)
    return c_void_p(t.data_ptr())


def darray(values):
    arr = (c_double * len(values))(*[float(v) for v in values])
    return arr


__all__ = ["load", "check", "Prior", "Bounds", "ptr", "stream_ptr", "darray", "require_cuda",
           "SIGNATURES", "LIB_PATH", "byref", "c_void_p", "c_int32", "c_int64", "c_double"]
