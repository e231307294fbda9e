"""ctypes binding of the C-ABI declared in ``include/wfcrl_b200.h`` (libwfcrl_b200.so, built in-tree by nvcc).

There is no CPU fallback: if the library cannot be loaded the import of any compute entry point fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

WF_MAX_TURBINES = 128
WF_TABLE_MAX = 64
WF_OK = 0
PREC_F64, PREC_F32 = 0, 1
KERNEL_BASIC, KERNEL_FAST = 0, 1
SHAPER_NONE, SHAPER_REFERENCE_PCT, SHAPER_STEP_PCT = 0, 1, 2


class WfConfig(C.Structure):
    _fields_ = [
        ("num_turbines", C.c_int32), ("num_envs", C.c_int32), ("device", C.c_int32), ("precision", C.c_int32),
        ("kernel", C.c_int32), ("max_iter", C.c_int32), ("continuous_control", C.c_int32),
        ("multi_agent", C.c_int32), ("reward_shaper", C.c_int32), ("fp32_relaxed", C.c_int32),
        ("yaw_lo", C.c_double), ("yaw_hi", C.c_double), ("yaw_step", C.c_double),
        ("load_coef", C.c_double), ("shaper_reference", C.c_double), ("dt", C.c_double),
        ("actuator_rate", C.c_double),
        ("air_density", C.c_double), ("turbulence_intensity", C.c_double), ("wind_shear", C.c_double),
        ("wind_veer", C.c_double),
        ("alpha", C.c_double), ("beta", C.c_double), ("ka", C.c_double), ("kb", C.c_double), ("ad", C.c_double),
        ("bd", C.c_double), ("dm", C.c_double),
        ("ch_initial", C.c_double), ("ch_constant", C.c_double), ("ch_ai", C.c_double), ("ch_downstream", C.c_double),
        ("rotor_diameter", C.c_double), ("hub_height", C.c_double), ("tsr", C.c_double), ("pP", C.c_double),
        ("pT", C.c_double), ("generator_efficiency", C.c_double), ("ref_density_cp_ct", C.c_double),
        ("table_len", C.c_int32), ("turbine_grid_points", C.c_int32),
        ("table_ws", C.c_double * WF_TABLE_MAX), ("table_cp", C.c_double * WF_TABLE_MAX),
        ("table_ct", C.c_double * WF_TABLE_MAX),
    ]


class WfStepOut(C.Structure):
    _fields_ = [
        ("yaw", C.c_void_p), ("wind_speed", C.c_void_p), ("wind_direction", C.c_void_p), ("power", C.c_void_p),
        ("load", C.c_void_p), ("reward", C.c_void_p), ("freewind", C.c_void_p), ("truncated", C.c_void_p),
    ]


# every symbol include/wfcrl_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "wf_default_config": (C.c_int, [C.POINTER(WfConfig)]),
    "wf_create": (C.c_int, [C.POINTER(WfConfig), _P, _P, C.POINTER(_P)]),
    "wf_destroy": (C.c_int, [_P]),
    "wf_set_layouts": (C.c_int, [_P, C.c_int32, _P, _P]),
    "wf_set_layouts_sized": (C.c_int, [_P, C.c_int32, _P, _P, _P]),
    "wf_assign_layouts": (C.c_int, [_P, _P, C.c_int32, _P, _P]),
    "wf_set_layout_sampling": (C.c_int, [_P, C.c_int32]),
    "wf_reset": (C.c_int, [_P, _P, C.c_int32, _P, _P, _P, _P, C.c_int32, C.POINTER(WfStepOut), _P]),
    "wf_reset_masked": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.POINTER(WfStepOut), _P]),
    "wf_reset_sampled": (C.c_int, [_P, _P, C.c_uint64, C.c_int64, C.c_double, C.c_double, C.c_int32, C.POINTER(WfStepOut), _P]),
    "wf_set_autoreset": (C.c_int, [_P, C.c_int32, C.c_uint64, C.c_int64, C.c_double, C.c_double]),
    "wf_autoreset_finish": (C.c_int, [_P, C.c_int32, C.POINTER(WfStepOut), _P]),
    "wf_set_kernel_timing": (C.c_int, [_P, C.c_int32]),
    "wf_get_kernel_timing": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "wf_step": (C.c_int, [_P, _P, C.POINTER(WfStepOut), _P]),
    "wf_update_command": (C.c_int, [_P, _P, C.POINTER(WfStepOut), _P]),
    "wf_evaluate_yaw": (C.c_int, [_P, _P, C.c_int32, _P, _P, _P]),
    "wf_evaluate_actions": (C.c_int, [_P, _P, C.c_int32, C.POINTER(WfStepOut), _P, _P]),
    "wf_evaluate_rollouts": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(WfStepOut), _P, _P]),
    "wf_step_host": (C.c_int, [_P, _P, C.POINTER(WfStepOut), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "wf_update_command_host": (C.c_int, [_P, _P, C.POINTER(WfStepOut)]),
    "wf_update_wind": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "wf_set_turbulence_intensity": (C.c_int, [_P, _P, _P]),
    "wf_get_state": (C.c_int, [_P, C.c_char_p, _P, C.c_size_t]),
    "wf_set_state": (C.c_int, [_P, C.c_char_p, _P, C.c_size_t]),
    "wf_device_info": (C.c_int, [_P] + [C.POINTER(C.c_int32)] * 6),
    "wf_launch_count": (C.c_uint64, [_P]),
    "wf_last_error": (C.c_char_p, []),
    "wf_version": (C.c_char_p, []),
}

_lib = None


class WfError(RuntimeError):
    pass


def library_path() -> str:
    return _build.LIB


def load():
    """Load (building in-tree first when nvcc is available and the .so is stale or missing)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if _build.needs_build():
        try:
            _build.build_library()
        except Exception as exc:  # no nvcc on this box: use the shipped .so if there is one
            if not os.path.exists(path):
                raise WfError(
                    "libwfcrl_b200.so is missing and could not be built (there is no CPU fallback): " + str(exc)
                ) from exc
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the ABI is incomplete
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def binary_matches_source() -> bool:
    """True when the loaded library reports the hash of the sources in the tree (wf_version vs build.source_hash)."""
    return load().wf_version().decode().endswith("wfcrl_b200-src-sha256:" + _build.source_hash())


def check(rc: int):
    if rc != WF_OK:
        raise WfError(f"wfcrl_b200 error {rc}: {load().wf_last_error().decode()}")
