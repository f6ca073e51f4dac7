"""ctypes binding of libgingr_cuda.so (the C ABI of include/gingr_cuda.h).

There is deliberately NO fallback: if the library is missing, or no B200 is present when a context is
created, the calls raise.  The CPU oracle (test infrastructure) is never imported here.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char, c_char_p, c_double, c_int32, c_int64, c_uint8, c_uint64, c_void_p

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# GINGR_CUDA_LIB: alternative build of the same library (kernel tuning experiments); never a fallback
LIB_PATH = os.environ.get("GINGR_CUDA_LIB") or os.path.join(HERE, "lib", "libgingr_cuda.so")

GINGR_OK = 0
GINGR_MODEL_FLEXIBILITY = 1
GINGR_ERR_ARG, GINGR_ERR_CUDA, GINGR_ERR_NCCL, GINGR_ERR_UNSUPPORTED = -1, -2, -3, -4

STATUS_NONE, STATUS_MAX_ITERATION, STATUS_CONVERGED, STATUS_MODEL_FLEXIBILITY_ERROR = 0, 1, 2, 3
SIMILARITY_TRANSFORMS, RIGID_TRANSFORMS, NO_TRANSFORMS = 0, 1, 2
TRIANGULAR_CLOSEST_POINT, ALONG_NORMAL_CLOSEST_POINT, POINTCLOUD_CLOSEST_POINT = 0, 1, 2
ALGO_CPD, ALGO_ICP = 0, 1


class GingrState(ctypes.Structure):
    """POD mirror of gingr_state (include/gingr_cuda.h)."""
    _fields_ = [
        ("scale", c_double),
        ("translation", c_double * 3),
        ("euler", c_double * 3),
        ("center", c_double * 3),
        ("sigma2", c_double),
        ("step_length", c_double),
        ("global_transformation", c_int32),
        ("iteration", c_int32),
        ("status", c_int32),
        ("rank", c_int32),
    ]


class GingrConfig(ctypes.Structure):
    """POD mirror of gingr_config (include/gingr_cuda.h)."""
    _fields_ = [
        ("algorithm", c_int32),
        ("max_iterations", c_int32),
        ("threshold", c_double),
        ("use_landmark_correspondence", c_int32),
        ("has_initial_sigma", c_int32),
        ("initial_sigma", c_double),
        ("w", c_double),
        ("lambda_", c_double),
        ("end_sigma", c_double),
        ("reverse_correspondence_direction", c_int32),
        ("correspondence_method", c_int32),
    ]


class GingrMcmcSettings(ctypes.Structure):
    """POD mirror of gingr_mcmc_settings (include/gingr_cuda.h)."""
    _fields_ = [
        ("random_mixture", c_double),
        ("uncertainty", c_double),
        ("evaluation_mode", c_int32),
        ("reserved", c_int32),
        ("rot_sdev", c_double * 3),
        ("trans_sdev", c_double * 3),
        ("shape_sdev", c_double * 3),
    ]


EVAL_MODEL_TO_TARGET, EVAL_TARGET_TO_MODEL, EVAL_SYMMETRIC = 0, 1, 2

dp = POINTER(c_double)
ip = POINTER(c_int32)
bp = POINTER(c_uint8)
vpp = POINTER(c_void_p)

# name -> (restype, argtypes).  Kept in the order of include/gingr_cuda.h; tests/test_abi.py checks
# that the header and this table agree and that the .so exports every symbol.
SIGNATURES = {
    "gingr_version": (c_int32, []),
    "gingr_ctx_create": (c_int32, [c_int32, vpp]),
    "gingr_ctx_destroy": (c_int32, [c_void_p]),
    "gingr_last_error": (c_char_p, [c_void_p]),
    "gingr_ctx_stream": (c_void_p, [c_void_p]),
    "gingr_ctx_synchronize": (c_int32, [c_void_p]),
    "gingr_ctx_launch_count": (c_int64, [c_void_p]),
    "gingr_comm_unique_id": (c_int32, [POINTER(c_char * 128)]),
    "gingr_comm_init": (c_int32, [c_void_p, c_int32, c_int32, POINTER(c_char * 128)]),
    "gingr_model_upload": (c_int32, [c_void_p, c_int32, c_int32, dp, dp, dp, c_int64, dp, ip, c_int32, vpp]),
    "gingr_model_destroy": (c_int32, [c_void_p]),
    "gingr_model_new_reference": (c_int32, [c_void_p, c_void_p, c_int32, dp, ip, c_int32, vpp]),
    "gingr_gpmm_gaussian_mixture": (c_int32, [c_void_p, c_int32, dp, ip, c_int32, c_int32, dp, dp, c_double, c_int32, vpp, ip]),
    "gingr_gpmm_gaussian_symmetric": (c_int32, [c_void_p, c_int32, dp, ip, c_int32, c_int32, dp, dp, c_double, c_int32, vpp, ip]),
    "gingr_gpmm_inverse_laplacian": (c_int32, [c_void_p, c_int32, dp, ip, c_int32, c_double, c_double, c_double, c_int32, vpp, ip]),
    "gingr_model_download": (c_int32, [c_void_p, c_void_p, ip, ip, dp, dp, dp, c_int64, dp]),
    "gingr_target_upload": (c_int32, [c_void_p, c_int32, dp, ip, c_int32, vpp]),
    "gingr_target_destroy": (c_int32, [c_void_p]),
    "gingr_cpd_estep": (c_int32, [c_void_p, c_void_p, c_int32, dp, c_double, c_double, dp, dp, dp]),
    "gingr_bcpd_estep": (c_int32, [c_void_p, c_void_p, c_int32, dp, dp, dp, c_double, c_double, c_double,
                                   dp, dp, dp, dp]),
    "gingr_cpd_initial_sigma2": (c_int32, [c_void_p, c_void_p, c_int32, dp, dp]),
    "gingr_icp_closest": (c_int32, [c_void_p, c_void_p, c_int32, dp, ip, c_int32, c_int32, ip, dp, bp, dp]),
    "gingr_icp_closest_reversal": (c_int32, [c_void_p, c_void_p, c_int32, dp, ip, c_int32, c_int32, ip, bp, dp]),
    "gingr_posterior_mean": (c_int32, [c_void_p, c_void_p, dp, dp, c_int32, ip, dp, c_int32, dp, dp, dp]),
    "gingr_posterior_covariance": (c_int32, [c_void_p, c_void_p, dp, dp, c_int32, ip, dp, c_int32, dp, dp]),
    "gingr_model_posterior": (c_int32, [c_void_p, c_void_p, dp, dp, c_int32, ip, dp, c_int32, dp, vpp]),
    "gingr_posterior_model_profile": (c_int32, [c_void_p, dp, ip]),
    "gingr_coefficients": (c_int32, [c_void_p, c_void_p, dp, dp, dp, dp]),
    "gingr_spd_solve": (c_int32, [c_void_p, c_int32, dp, c_int32, dp, dp, dp, dp, c_int32, dp]),
    "gingr_model_instance": (c_int32, [c_void_p, c_void_p, POINTER(GingrState), dp, dp]),
    "gingr_registration_create": (c_int32, [c_void_p, c_void_p, c_void_p, POINTER(GingrConfig), vpp]),
    "gingr_registration_destroy": (c_int32, [c_void_p]),
    "gingr_registration_set_landmarks": (c_int32, [c_void_p, c_int32, ip, dp, dp]),
    "gingr_initialize_state": (c_int32, [c_void_p, POINTER(GingrState), dp, dp]),
    "gingr_update": (c_int32, [c_void_p, POINTER(GingrState), dp, c_int32, c_uint64, POINTER(GingrState), dp, dp]),
    "gingr_update_chain": (c_int32, [c_void_p, c_int32]),
    "gingr_update_chain_sampled": (c_int32, [c_void_p, c_int32, c_uint64]),
    "gingr_update_batch": (c_int32, [POINTER(c_void_p), c_int32, c_int32, c_int32, c_uint64]),
    "gingr_state_download": (c_int32, [c_void_p, POINTER(GingrState), dp, dp]),
    "gingr_registration_posterior_model": (c_int32, [c_void_p, POINTER(GingrState), dp, vpp]),
    "gingr_mcmc_configure": (c_int32, [c_void_p, POINTER(GingrMcmcSettings), ip, c_int32, ip, c_int32]),
    "gingr_evaluate_log_value": (c_int32, [c_void_p, POINTER(GingrState), dp, dp]),
    "gingr_log_transition_probability": (c_int32, [c_void_p, POINTER(GingrState), dp, POINTER(GingrState), dp, dp]),
    "gingr_mcmc_chain": (c_int32, [c_void_p, c_int32, c_uint64]),
    "gingr_mcmc_batch": (c_int32, [POINTER(c_void_p), c_int32, c_int32, c_uint64]),
    "gingr_mcmc_stats": (c_int32, [c_void_p, dp, ip]),
    "gingr_mcmc_best": (c_int32, [c_void_p, POINTER(GingrState), dp, dp]),
    "gingr_registration_set_profiling": (c_int32, [c_void_p, c_int32]),
    "gingr_registration_get_profile": (c_int32, [c_void_p, dp, ip]),
}

_lib = None


class GingrError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libgingr_cuda error {code}: {msg}")
        self.code = code


def load(bind: bool = True):
    """Load libgingr_cuda.so.  Raises if the library has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GingrError(GINGR_ERR_CUDA, f"{LIB_PATH} not found -- build it with `python -m gingr_b200.build` "
                         "(the hot path is CUDA only; there is no CPU fallback)")
    lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
    if bind:
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name, None)
            if fn is None:   # stale build: calling it raises, nothing is emulated
                raise GingrError(GINGR_ERR_UNSUPPORTED, f"{LIB_PATH} does not export {name}; rebuild it")
            fn.restype = res
            fn.argtypes = args
    _lib = lib
    return lib


def check(code: int, ctx=None) -> int:
    if code < 0:
        msg = load().gingr_last_error(ctx)
        raise GingrError(code, msg.decode() if msg else "")
    return code


def as_dp(a):
    return None if a is None else a.ctypes.data_as(dp)


def as_ip(a):
    return None if a is None else a.ctypes.data_as(ip)


def as_bp(a):
    return None if a is None else a.ctypes.data_as(bp)


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)
