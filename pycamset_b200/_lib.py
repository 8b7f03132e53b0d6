"""ctypes binding of libpcs_b200.so (the C ABI declared in include/pcs_b200.h).

The library is the product path: if it cannot be loaded, or no CUDA device works, every call raises.
There is no CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as ct
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libpcs_b200.so"

PCS_OK = 0
PCS_ERR_INVALID, PCS_ERR_CHAIN, PCS_ERR_CUDA, PCS_ERR_UNSUPPORTED, PCS_ERR_NUMERIC = -1, -2, -3, -4, -5
CHAIN_TEMPLATE, CHAIN_SELFCAL = 0, 1
PRECISION_FP64, PRECISION_MIXED = 0, 1

EXPORTED_SYMBOLS = [
    "pcs_chain_from_name", "pcs_problem_create", "pcs_problem_destroy", "pcs_problem_get_info", "pcs_last_error",
    "pcs_set_param_string", "pcs_set_free", "pcs_get_param_string", "pcs_residual", "pcs_residual_dev",
    "pcs_csr_structure", "pcs_jacobian_values", "pcs_jacobian_values_dev", "pcs_segments", "pcs_normal_equations",
    "pcs_normal_equations_dev", "pcs_point_blocks", "pcs_normal_dense", "pcs_device_buffers_get", "pcs_set_allreduce",
    "pcs_lm_default_options", "pcs_lm_solve", "pcs_covariance", "pcs_spd_solve", "pcs_syrk_sub", "pcs_lm_schur_fraction", "pcs_timing_enable", "pcs_timing_get", "pcs_timing_get_all", "pcs_launch_count",
    "pcs_costfn", "pcs_gauge_scale", "pcs_set_normal_precision", "pcs_p2p_buffer_bytes", "pcs_p2p_allreduce_setup", "pcs_p2p_allreduce_camera_blocks", "pcs_p2p_status", "pcs_device_sm_count",
    "pcs_version",
]


class PcsError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"pcs_b200 error {code}: {message}")
        self.code = code


class UnknownChainError(PcsError, ValueError):
    """Raised for function-block chains that have no CUDA kernel (the GPU path never falls back to the CPU)."""


class ProblemDesc(ct.Structure):
    _fields_ = [
        ("chain", ct.c_int32), ("device", ct.c_int32), ("n_obs", ct.c_int64), ("n_cams", ct.c_int32),
        ("n_poses", ct.c_int32), ("n_keys", ct.c_int32), ("inputs_on_device", ct.c_int32),
        ("cam", ct.c_void_p), ("pose", ct.c_void_p), ("key", ct.c_void_p), ("uv", ct.c_void_p),
        ("template_xyz", ct.c_void_p), ("free_map", ct.c_void_p), ("stream", ct.c_void_p),
    ]


class ProblemInfo(ct.Structure):
    _fields_ = [
        ("chain", ct.c_int32), ("n_cams", ct.c_int32), ("n_poses", ct.c_int32), ("n_keys", ct.c_int32),
        ("cols_per_row", ct.c_int32), ("device", ct.c_int32), ("n_obs", ct.c_int64), ("n_params", ct.c_int64),
        ("n_free", ct.c_int64), ("nnz", ct.c_int64), ("n_segments", ct.c_int64),
    ]


class DeviceBuffers(ct.Structure):
    _fields_ = [(n, ct.c_void_p) for n in ("params", "U", "gc", "V", "gp", "W", "cost", "residual", "stream")]


class LmOptions(ct.Structure):
    _fields_ = [
        ("max_iter", ct.c_int32), ("verbose", ct.c_int32), ("lambda0", ct.c_double), ("ftol", ct.c_double),
        ("xtol", ct.c_double), ("gtol", ct.c_double), ("lambda_min", ct.c_double), ("lambda_max", ct.c_double),
    ]


class LmStats(ct.Structure):
    _fields_ = [
        ("iterations", ct.c_int32), ("n_eval_normal", ct.c_int32), ("n_eval_cost", ct.c_int32), ("status", ct.c_int32),
        ("cost_initial", ct.c_double), ("cost_final", ct.c_double), ("grad_norm_inf", ct.c_double),
        ("lambda_final", ct.c_double), ("seconds", ct.c_double),
    ]


ALLREDUCE_FN = ct.CFUNCTYPE(ct.c_int, ct.c_void_p, ct.c_void_p, ct.c_int64, ct.c_int, ct.c_void_p)

_lib = None


def load() -> ct.CDLL:
    """Load the CUDA library; raise loudly when it is missing (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m pycamset_b200.build` (or __graft_entry__.build()); "
            "pycamset_b200 has no CPU fallback")
    lib = ct.CDLL(str(LIB_PATH))
    vp, i64p = ct.c_void_p, ct.POINTER(ct.c_int64)
    lib.pcs_last_error.restype = ct.c_char_p
    lib.pcs_version.restype = ct.c_char_p
    lib.pcs_chain_from_name.argtypes = [ct.c_char_p]
    lib.pcs_problem_create.argtypes = [ct.POINTER(ProblemDesc), ct.POINTER(vp)]
    lib.pcs_problem_destroy.argtypes = [vp]
    lib.pcs_problem_get_info.argtypes = [vp, ct.POINTER(ProblemInfo)]
    lib.pcs_set_param_string.argtypes = [vp, vp]
    lib.pcs_set_free.argtypes = [vp, vp]
    lib.pcs_get_param_string.argtypes = [vp, vp]
    lib.pcs_residual.argtypes = [vp, vp, vp]
    lib.pcs_residual_dev.argtypes = [vp, vp, vp]
    lib.pcs_csr_structure.argtypes = [vp, vp, vp]
    lib.pcs_jacobian_values.argtypes = [vp, vp, vp]
    lib.pcs_jacobian_values_dev.argtypes = [vp, vp, vp]
    lib.pcs_segments.argtypes = [vp, vp, vp, vp]
    lib.pcs_normal_equations.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    lib.pcs_normal_equations_dev.argtypes = [vp, vp]
    lib.pcs_point_blocks.argtypes = [vp, vp, vp, vp, vp]
    lib.pcs_normal_dense.argtypes = [vp, vp, vp, vp, vp]
    lib.pcs_device_buffers_get.argtypes = [vp, ct.POINTER(DeviceBuffers)]
    lib.pcs_set_allreduce.argtypes = [vp, ALLREDUCE_FN, vp, ct.c_int, ct.c_int]
    lib.pcs_lm_default_options.argtypes = [ct.POINTER(LmOptions)]
    lib.pcs_lm_solve.argtypes = [vp, vp, ct.POINTER(LmOptions), vp, ct.POINTER(LmStats)]
    lib.pcs_covariance.argtypes = [vp, vp, vp, vp, vp, ct.POINTER(ct.c_double), i64p]
    lib.pcs_spd_solve.argtypes = [ct.c_int, ct.c_int64, vp, vp, vp, ct.POINTER(ct.c_int)]
    lib.pcs_syrk_sub.argtypes = [ct.c_int, ct.c_int64, ct.c_int64, vp, vp]
    lib.pcs_lm_schur_fraction.argtypes = [vp, ct.POINTER(ct.c_double)]
    lib.pcs_timing_enable.argtypes = [vp, ct.c_int]
    lib.pcs_timing_get.argtypes = [vp, ct.POINTER(ct.c_double)]
    lib.pcs_timing_get_all.argtypes = [vp, vp, ct.c_int64, ct.POINTER(ct.c_int64)]
    lib.pcs_launch_count.argtypes = [vp, ct.POINTER(ct.c_int64)]
    lib.pcs_set_normal_precision.argtypes = [vp, ct.c_int]
    lib.pcs_gauge_scale.argtypes = [ct.c_int, ct.c_int64, vp, vp, vp, ct.c_double, ct.c_double, ct.c_double, ct.POINTER(ct.c_double), ct.POINTER(ct.c_int64)]
    lib.pcs_costfn.argtypes = [vp, ct.c_int, vp, vp, vp, vp, vp, vp]
    lib.pcs_p2p_buffer_bytes.argtypes = [vp, ct.c_int]
    lib.pcs_p2p_status.argtypes = [vp, ct.POINTER(ct.c_int)]
    lib.pcs_p2p_buffer_bytes.restype = ct.c_int64
    lib.pcs_p2p_allreduce_setup.argtypes = [vp, ct.c_int, ct.c_int, ct.POINTER(vp), ct.c_int64]
    lib.pcs_p2p_allreduce_camera_blocks.argtypes = [vp]
    lib.pcs_device_sm_count.argtypes = [ct.c_int]
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc == PCS_OK:
        return
    msg = load().pcs_last_error().decode(errors="replace")
    if rc == PCS_ERR_CHAIN:
        raise UnknownChainError(rc, msg)
    raise PcsError(rc, msg)
