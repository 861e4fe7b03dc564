"""dcmrta_b200/_lib.py -- ctypes binding of include/dcmrta.h (the C ABI of libdcmrta_b200.so).

The product path has no CPU fallback: if the CUDA library cannot be loaded, or a call fails, a DcmError is raised.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

from . import build as _build

_LIB = None

STATUS = {0: "DCM_OK", -1: "DCM_ERR_ARG", -2: "DCM_ERR_SHAPE", -3: "DCM_ERR_DEVICE", -4: "DCM_ERR_CUDA", -5: "DCM_ERR_STATE",
          -6: "DCM_ERR_NOMEM"}

FLAG_AUTO_RESET, FLAG_REGENERATE, FLAG_INDIVIDUAL = 1, 2, 4
PROTOCOL = {"LF": 0, "IA": FLAG_INDIVIDUAL}     # leader-follower (worker.py:45-85) / individual agent (worker.py:159-198)
POLICY = {"external": 0, "random": 1, "greedy": 2}
ENV_DONE, ENV_FINISHED, ENV_STUCK = 1, 2, 4
ENV_ERR_OVERFLOW, ENV_ERR_ACTION, ENV_ERR_FOLLOW, ENV_ERR_LEADER = 16, 32, 64, 128
ENV_ERR_MASK = ENV_ERR_OVERFLOW | ENV_ERR_ACTION | ENV_ERR_FOLLOW | ENV_ERR_LEADER


class DcmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"{STATUS.get(code, code)}: {msg}")
        self.code = code


vp, i32, u32, u64, f64, sz = C.c_void_p, C.c_int, C.c_uint32, C.c_uint64, C.c_double, C.c_size_t

# name -> (restype, argtypes); every symbol include/dcmrta.h declares
SIGNATURES = {
    "dcm_create": (i32, [C.POINTER(vp), i32, i32, i32, i32, i32, u32]),
    "dcm_destroy": (i32, [vp]),
    "dcm_set_params": (i32, [vp, f64, f64, f64]),
    "dcm_seed": (i32, [vp, u64, u64]),
    "dcm_load_instances": (i32, [vp, vp, vp, vp, vp, vp]),
    "dcm_load_instances_host": (i32, [vp, vp, vp, vp, vp]),
    "dcm_generate": (i32, [vp, f64, i32, vp]),
    "dcm_get_instances": (i32, [vp, vp, vp, vp, vp, vp]),
    "dcm_reset": (i32, [vp, vp, vp, vp, vp, vp, vp, vp]),
    "dcm_step": (i32, [vp, vp, vp, i32, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp]),
    "dcm_step_host": (i32, [vp, vp, i32, vp, vp, vp, vp, vp, vp]),
    "dcm_episode_metrics": (i32, [vp, vp, vp]),
    "dcm_next_decision": (i32, [vp, vp, vp, vp]),
    "dcm_unique_group": (i32, [vp, vp, vp, vp]),
    "dcm_set_clock": (i32, [vp, vp, vp]),
    "dcm_get_clock": (i32, [vp, vp, vp]),
    "dcm_task_update": (i32, [vp, vp, vp]),
    "dcm_agent_update": (i32, [vp, vp]),
    "dcm_apply_members": (i32, [vp, vp, vp, i32, vp, vp, vp]),
    "dcm_build_obs": (i32, [vp, vp, vp, vp, vp, vp]),
    "dcm_check_finished": (i32, [vp, vp, vp]),
    "dcm_compute_metrics": (i32, [vp, vp, vp, vp, vp]),
    "dcm_execute_by_route": (i32, [vp, vp, i32, vp, vp, vp]),
    "dcm_record_bytes": (sz, [vp]),
    "dcm_export_state": (i32, [vp, vp, sz, vp]),
    "dcm_import_state": (i32, [vp, vp, sz, vp]),
    "dcm_layout": (i32, [vp, vp, i32]),
    "dcm_env_flags": (i32, [vp, vp, vp]),
    "dcm_total_steps": (i32, [vp, C.POINTER(u64)]),
    "dcm_total_episodes": (i32, [vp, C.POINTER(u64)]),
    "dcm_algorithmic_bytes_per_step": (sz, [vp]),
    "dcm_launch_count": (u64, [vp]),
    "dcm_debug_pass_trace": (i32, [vp, vp, sz]),
    "dcm_last_error": (C.c_char_p, []),
    "dcm_version": (C.c_char_p, []),
}


def library_path() -> Path:
    return _build.SO


def lib() -> C.CDLL:
    """Load libdcmrta_b200.so (building it in-tree first when it is missing or stale and nvcc is present)."""
    global _LIB
    if _LIB is None:
        try:
            so = _build.build()
        except Exception as e:                     # no nvcc: a prebuilt, up-to-date .so is still fine
            so = _build.SO
            if not so.exists():
                raise DcmError(-3, f"libdcmrta_b200.so is missing and cannot be built ({e}); there is no CPU fallback")
        L = C.CDLL(str(so))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _LIB = L
    return _LIB


def check(rc: int):
    if rc != 0:
        raise DcmError(rc, lib().dcm_last_error().decode())
