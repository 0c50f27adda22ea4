"""Recompute mode (include/dpb200.h: pi_create, DPB200_TABLE) on a machine without a GPU: the builder program, which now
also holds pi_improve_recompute and pi_policy_rows, compiles for sm_100a against every plugin's dynamics, compile
errors carry the NVRTC log, and the new entry points are bound with the header's signatures."""
import ctypes as C
import importlib.util
import re
from pathlib import Path

import pytest

from dynamicprogramming_b200 import _ffi, compat, envs

ROOT = Path(__file__).resolve().parents[1]
FIXTURE = ROOT / "tests" / "fixtures" / "double_integrator_cuda.py"
_spec = importlib.util.spec_from_file_location("odd_dims", ROOT / "tests" / "fixtures" / "odd_dims.py")
odd = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(odd)


def _plugin_src(name: str) -> str:
    spec = envs.REGISTRY[name]
    inst = spec.cls.__new__(spec.cls)
    for k, v in spec.kwargs.items():
        setattr(inst, k, v)
    return inst._dynamics_cuda_src()


def _compile(src: str, D: int) -> int:
    n = C.c_int64()
    _ffi.check(_ffi.lib().pi_recompute_compile_check(src.encode(), D, C.byref(n)))
    return n.value


@pytest.mark.parametrize("name", sorted(envs.REGISTRY))
def test_recompute_kernels_compile_for_every_plugin(name):
    assert _compile(_plugin_src(name), envs.REGISTRY[name].cls.N_DIMS) > 1000


@pytest.mark.parametrize("D", [1, 2, 3, 4, 5, 6])
def test_recompute_kernels_compile_for_the_odd_dims_fixture(D):
    assert _compile(odd.dynamics_src(D), D) > 1000


def test_recompute_kernels_compile_for_the_reference_style_fixture():
    g = compat.load_runner(FIXTURE)
    compat.uninstall()
    cls = g["DoubleIntegratorCuda"]
    assert _compile(cls.__new__(cls)._dynamics_cuda_src(), 2) > 1000


def test_compile_errors_carry_the_nvrtc_log():
    lib = _ffi.lib()
    bad = "__device__ void step_dynamics(float a, float b, float u, float* x, float* y, float* r, bool* t) { oops; }"
    assert lib.pi_recompute_compile_check(bad.encode(), 2, None) == _ffi.PI_ERR_COMPILE
    msg = lib.pi_last_error().decode()
    assert "oops" in msg and "error" in msg.lower()
    assert lib.pi_recompute_compile_check(_plugin_src("pendulum").encode(), 4, None) == _ffi.PI_ERR_COMPILE
    assert "PI_CALL_STEP_DYNAMICS" in lib.pi_last_error().decode()
    assert lib.pi_recompute_compile_check(None, 2, None) == _ffi.PI_ERR_INVALID
    assert lib.pi_recompute_compile_check(b"", 0, None) == _ffi.PI_ERR_INVALID


def test_bindings_match_the_header():
    header = (ROOT / "include" / "dpb200.h").read_text()
    assert re.search(r"int32_t pi_table_mode\(const pi_engine\* e\);", header)
    assert re.search(r"int pi_recompute_compile_check\(const char\* dynamics_src, int32_t n_dims, int64_t\* cubin_bytes\);",
                     header)
    restype, args = _ffi.SIGNATURES["pi_table_mode"]
    assert restype is C.c_int32 and args == [C.c_void_p]
    restype, args = _ffi.SIGNATURES["pi_recompute_compile_check"]
    assert restype is C.c_int and args == [C.c_char_p, C.c_int32, C.POINTER(C.c_int64)]
    lib = _ffi.lib()
    assert lib.pi_table_mode(None) == 0
    assert lib.pi_table_bytes(None) == 0
