"""ctypes binding of libcudampc.so (include/cudampc.h).  No fallback: a missing library is an ImportError
with build instructions, a failing CUDA call is a RuntimeError carrying cudampc_last_error()."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CUDAMPC_LIB") or os.path.join(_HERE, "libcudampc.so")      # CUDAMPC_LIB: dev builds (timing, poison)


class Params(C.Structure):
    _fields_ = [("wheelbase_px", C.c_double), ("dt", C.c_double), ("horizon", C.c_int32), ("_pad", C.c_int32),
                ("q", C.c_double * 16), ("r", C.c_double * 4), ("q_terminal", C.c_double * 16),
                ("u_bounds", C.c_double * 4), ("v_bounds", C.c_double * 2), ("du_bounds", C.c_double * 4),
                ("slack_velocity", C.c_double), ("slack_input", C.c_double), ("slack_rate", C.c_double)]


# the same record as a NumPy structured dtype (arrays of per-problem parameters, field-wise editable: arr["du_bounds"][:, 3] = ...)
PARAMS_DTYPE = np.dtype([(name, np.float64 if t is C.c_double else np.int32 if t is C.c_int32 else (np.float64, (t._length_,)))
                         for name, t in Params._fields_], align=True)
assert PARAMS_DTYPE.itemsize == C.sizeof(Params)

# status of a problem whose own parameter record was rejected (CUDAMPC_INVALID_PARAMS)
STATUS_INVALID_PARAMS = -100


class Settings(C.Structure):
    _fields_ = [("eps_abs", C.c_double), ("eps_rel", C.c_double), ("rho", C.c_double), ("alpha", C.c_double),
                ("sigma", C.c_double), ("adaptive_rho_tolerance", C.c_double), ("rho_eq_factor", C.c_double),
                ("rho_min", C.c_double), ("rho_max", C.c_double), ("delta", C.c_double),
                ("max_iter", C.c_int32), ("check_termination", C.c_int32), ("adaptive_rho", C.c_int32),
                ("adaptive_rho_interval", C.c_int32), ("polish_passes", C.c_int32), ("polish_refine_iter", C.c_int32),
                ("warm_start", C.c_int32), ("polish_retry", C.c_int32),
                ("early_polish", C.c_int32), ("early_polish_start", C.c_int32)]


class RolloutCfg(C.Structure):
    _fields_ = [("sim_steps", C.c_int32), ("relax_on_failure", C.c_int32), ("advance_dist2", C.c_double),
                ("goal_radius", C.c_double), ("relax_v_scale", C.c_double), ("relax_da", C.c_double),
                ("relax_ddelta", C.c_double), ("step_ns_dev", C.c_void_p)]


# every symbol include/cudampc.h declares (tests/test_abi.py checks the library exports all of them)
SYMBOLS = (
    "cudampc_version", "cudampc_default_settings", "cudampc_default_rollout_cfg", "cudampc_create",
    "cudampc_destroy", "cudampc_last_error", "cudampc_set_params", "cudampc_linearize_batch", "cudampc_f_discrete_batch",
    "cudampc_solve_batch", "cudampc_solve_batch_host", "cudampc_build_reference_batch", "cudampc_rollout_batch",
    "cudampc_track_step_batch", "cudampc_solve_batch_params", "cudampc_rollout_batch_params", "cudampc_track_step_batch_params",
    "cudampc_workspace_doubles",
    "cudampc_problems_per_sm", "cudampc_rollout_resident", "cudampc_launch_count", "cudampc_fp64_peak_tflops",
)

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU fallback for the MPC hot path.")
    lib = C.CDLL(LIB_PATH)
    vp, dp, ip = C.c_void_p, C.c_void_p, C.c_void_p
    lib.cudampc_version.restype = C.c_int
    lib.cudampc_default_settings.argtypes = [C.POINTER(Settings)]
    lib.cudampc_default_settings.restype = None
    lib.cudampc_default_rollout_cfg.argtypes = [C.POINTER(RolloutCfg)]
    lib.cudampc_default_rollout_cfg.restype = None
    lib.cudampc_create.argtypes = [C.POINTER(Params), C.c_int, C.c_int, C.POINTER(vp)]
    lib.cudampc_create.restype = C.c_int
    lib.cudampc_destroy.argtypes = [vp]
    lib.cudampc_destroy.restype = C.c_int
    lib.cudampc_last_error.argtypes = [vp]
    lib.cudampc_last_error.restype = C.c_char_p
    lib.cudampc_set_params.argtypes = [vp, C.POINTER(Params)]
    lib.cudampc_set_params.restype = C.c_int
    lib.cudampc_linearize_batch.argtypes = [vp, C.c_int, dp, dp, dp, dp, vp]
    lib.cudampc_linearize_batch.restype = C.c_int
    lib.cudampc_f_discrete_batch.argtypes = [vp, C.c_int, dp, dp, dp, dp, vp]
    lib.cudampc_f_discrete_batch.restype = C.c_int
    solve_args = [vp, C.c_int, dp, dp, dp, C.POINTER(Settings), dp, dp, dp, ip, ip, dp, dp, ip, vp]
    lib.cudampc_solve_batch.argtypes = solve_args
    lib.cudampc_solve_batch.restype = C.c_int
    lib.cudampc_solve_batch_host.argtypes = solve_args
    lib.cudampc_solve_batch_host.restype = C.c_int
    lib.cudampc_build_reference_batch.argtypes = [vp, C.c_int, dp, ip, C.c_int, C.c_double, dp, ip, C.c_int, vp]
    lib.cudampc_build_reference_batch.restype = C.c_int
    lib.cudampc_rollout_batch.argtypes = [vp, C.c_int, dp, ip, C.c_int, dp, dp, C.POINTER(Settings),
                                          C.POINTER(RolloutCfg), dp, dp, ip, ip, ip, ip, vp]
    lib.cudampc_rollout_batch.restype = C.c_int
    lib.cudampc_track_step_batch.argtypes = [vp, C.c_int, dp, ip, C.c_int, dp, dp, C.POINTER(Settings), C.POINTER(RolloutCfg),
                                             ip, dp, ip, ip, dp, dp, dp, ip, ip, vp]
    lib.cudampc_track_step_batch.restype = C.c_int
    lib.cudampc_solve_batch_params.argtypes = [vp, C.c_int, dp, dp, dp, C.POINTER(Settings), vp, dp, dp, dp, ip, ip, dp, dp, ip, vp]
    lib.cudampc_solve_batch_params.restype = C.c_int
    lib.cudampc_rollout_batch_params.argtypes = [vp, C.c_int, dp, ip, C.c_int, dp, dp, C.POINTER(Settings),
                                                 C.POINTER(RolloutCfg), vp, dp, dp, ip, ip, ip, ip, vp]
    lib.cudampc_rollout_batch_params.restype = C.c_int
    lib.cudampc_track_step_batch_params.argtypes = [vp, C.c_int, dp, ip, C.c_int, dp, dp, C.POINTER(Settings), C.POINTER(RolloutCfg),
                                                    vp, ip, dp, ip, ip, dp, dp, dp, ip, ip, vp]
    lib.cudampc_track_step_batch_params.restype = C.c_int
    lib.cudampc_workspace_doubles.argtypes = [vp]
    lib.cudampc_workspace_doubles.restype = C.c_int
    lib.cudampc_problems_per_sm.argtypes = [vp]
    lib.cudampc_problems_per_sm.restype = C.c_int
    lib.cudampc_rollout_resident.argtypes = [vp]
    lib.cudampc_rollout_resident.restype = C.c_int
    lib.cudampc_launch_count.argtypes = [vp]
    lib.cudampc_launch_count.restype = C.c_int64
    lib.cudampc_fp64_peak_tflops.argtypes = [vp]
    lib.cudampc_fp64_peak_tflops.restype = C.c_double
    _lib = lib
    return lib


def check(lib, handle, rc: int, what: str) -> None:
    if rc != 0:
        msg = lib.cudampc_last_error(handle)
        raise RuntimeError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")
