"""
ctypes binding of libdpb200.so (the C ABI in include/dpb200.h).

There is deliberately no fallback: if the shared library is missing or cannot
be loaded, importing the engine raises, and pi_create fails without a CUDA
device.  Nothing here imports anything from oracle/.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

PI_MAX_DIMS = 6
PI_OK = 0
PI_ERR_INVALID, PI_ERR_CUDA, PI_ERR_COMPILE, PI_ERR_COMM, PI_ERR_NO_DEVICE = 1, 2, 3, 4, 5
PI_ROW_TERMINATED = -1
PI_ROW_ABSORBING = -2

_LIB_PATH = Path(os.environ.get("DPB200_LIB", Path(__file__).resolve().parent / "libdpb200.so"))


class PiGrid(C.Structure):
    _fields_ = [
        ("n_dims", C.c_int32),
        ("shape", C.c_int32 * PI_MAX_DIMS),
        ("lo", C.c_float * PI_MAX_DIMS),
        ("hi", C.c_float * PI_MAX_DIMS),
        ("axes", C.POINTER(C.c_float) * PI_MAX_DIMS),
    ]


class PiConfig(C.Structure):
    _fields_ = [
        ("gamma", C.c_float),
        ("theta", C.c_float),
        ("max_eval_iter", C.c_int32),
        ("max_pi_iter", C.c_int32),
        ("log_interval", C.c_int32),
        ("sync_interval", C.c_int32),
    ]


class PiShard(C.Structure):
    _fields_ = [
        ("rank", C.c_int32),
        ("world_size", C.c_int32),
        ("nccl_id", C.c_uint8 * 128),
    ]


class PiStats(C.Structure):
    _fields_ = [
        ("pi_iterations", C.c_int32),
        ("converged", C.c_int32),
        ("eval_sweeps", C.c_int64),
        ("last_delta", C.c_float),
        ("last_changed", C.c_int64),
        ("build_ms", C.c_double),
        ("eval_ms", C.c_double),
        ("improve_ms", C.c_double),
    ]

    def as_dict(self) -> dict:
        return {name: getattr(self, name) for name, _ in self._fields_}


LOG_FN = C.CFUNCTYPE(None, C.c_int, C.c_char_p, C.c_void_p)

# name -> (restype, argtypes); this table is also what the CPU test-suite checks
# against include/dpb200.h.
SIGNATURES = {
    "pi_last_error": (C.c_char_p, []),
    "pi_abi_version": (C.c_int, []),
    "pi_device_count": (C.c_int, []),
    "pi_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "pi_nvrtc_counters": (C.c_int, [C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "pi_compile_check": (C.c_int, [C.c_char_p, C.c_int32, C.POINTER(C.c_int64)]),
    "pi_create": (C.c_int, [C.POINTER(PiGrid), C.POINTER(C.c_float), C.c_int32, C.POINTER(PiConfig), C.c_char_p,
                            C.c_int32, C.POINTER(PiShard), C.POINTER(C.c_void_p)]),
    "pi_destroy": (None, [C.c_void_p]),
    "pi_set_log": (C.c_int, [C.c_void_p, LOG_FN, C.c_void_p]),
    "pi_set_terminal": (C.c_int, [C.c_void_p, C.c_void_p, C.c_float]),
    "pi_set_values": (C.c_int, [C.c_void_p, C.c_void_p, C.c_float]),
    "pi_set_values_buffer": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_float]),
    "pi_build_table": (C.c_int, [C.c_void_p]),
    "pi_retrain": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_float, C.POINTER(C.c_int32)]),
    "pi_evaluate": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int32)]),
    "pi_improve": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    "pi_run": (C.c_int, [C.c_void_p, C.POINTER(PiStats)]),
    "pi_copy_results": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "pi_copy_local_results": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "pi_upload_policy": (C.c_int, [C.c_void_p, C.c_void_p]),
    "pi_upload_values": (C.c_int, [C.c_void_p, C.c_void_p]),
    "pi_upload_policy_local": (C.c_int, [C.c_void_p, C.c_void_p]),
    "pi_sweeps": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "pi_expand_rows": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p]),
    "pi_device_ptrs": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                 C.POINTER(C.c_void_p)]),
    "pi_layout": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_double)]),
    "pi_n_states": (C.c_int64, [C.c_void_p]),
    "pi_local_begin": (C.c_int64, [C.c_void_p]),
    "pi_local_end": (C.c_int64, [C.c_void_p]),
    "pi_table_bytes": (C.c_int64, [C.c_void_p]),
    "pi_launch_count": (C.c_int64, [C.c_void_p]),
    "pi_get_stats": (C.c_int, [C.c_void_p, C.POINTER(PiStats)]),
    "pi_lookup_actions": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "pi_prolong_values": (C.c_int, [C.c_void_p, C.POINTER(PiGrid), C.c_void_p, C.POINTER(C.c_float)]),
    "pi_lookup_create": (C.c_int, [C.POINTER(PiGrid), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]),
    "pi_lookup_query": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "pi_lookup_destroy": (None, [C.c_void_p]),
    "pi_rollout_create": (C.c_int, [C.POINTER(PiGrid), C.c_void_p, C.c_void_p, C.c_int32, C.c_char_p, C.c_int32,
                                    C.POINTER(C.c_void_p)]),
    "pi_rollout_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pi_rollout_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pi_rollout_destroy": (None, [C.c_void_p]),
    "pi_rollout_compile_check": (C.c_int, [C.c_char_p, C.c_int32, C.POINTER(C.c_int64)]),
    "pi_eval_kernel_info": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "pi_xline_compile_check": (C.c_int, [C.c_int32, C.c_int32, C.c_char_p, C.POINTER(C.c_int64)]),
    "pi_debug_pair": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "pi_debug_plane": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                 C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "pi_debug_xline": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                 C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
}

_lib = None


class EngineError(RuntimeError):
    """Raised for every non-zero status of the C ABI (the reference raises
    RuntimeError / cupy CompileException in the same places)."""

    def __init__(self, code: int, message: str) -> None:
        super().__init__(f"[dpb200 error {code}] {message}")
        self.code = code


def lib() -> C.CDLL:
    """Load libdpb200.so (once).  Fails loudly if the CUDA extension is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise RuntimeError(
            f"{_LIB_PATH} not found: the B200 engine has no CPU fallback. "
            "Build it with `python -m dynamicprogramming_b200.build` (needs nvcc)."
        )
    handle = C.CDLL(str(_LIB_PATH), mode=C.RTLD_GLOBAL)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(handle, name)  # AttributeError if the symbol is missing
        fn.restype = restype
        fn.argtypes = argtypes
    if handle.pi_abi_version() != 1:
        raise RuntimeError("libdpb200.so ABI version mismatch")
    _lib = handle
    return handle


def check(rc: int) -> None:
    if rc != PI_OK:
        raise EngineError(rc, lib().pi_last_error().decode(errors="replace"))


def ptr(a: np.ndarray) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data)
