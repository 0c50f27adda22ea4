"""N5 closed-loop rollouts (include/dpb200.h: pi_rollout_*) on a box without a GPU: the rollout kernels compile for
sm_100a against every plugin's dynamics, compile errors carry the NVRTC log, compiles go through the disk cache, and
there is no CPU fallback."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from dynamicprogramming_b200 import _ffi, compat, envs, runners

FIXTURE = Path(__file__).resolve().parent / "fixtures" / "double_integrator_cuda.py"


def _plugin_src(name: str) -> str:
    spec = envs.REGISTRY[name]
    inst = spec.cls.__new__(spec.cls)
    for k, v in spec.kwargs.items():
        setattr(inst, k, v)
    return inst._dynamics_cuda_src()


def _compile(src: str, D: int) -> int:
    n = C.c_int64()
    _ffi.check(_ffi.lib().pi_rollout_compile_check(src.encode(), D, C.byref(n)))
    return n.value


@pytest.mark.parametrize("name", sorted(envs.REGISTRY))
def test_rollout_kernels_compile_for_every_plugin(name):
    assert _compile(_plugin_src(name), envs.REGISTRY[name].cls.N_DIMS) > 1000


def test_rollout_kernels_compile_for_the_reference_style_fixture():
    g = compat.load_runner(FIXTURE)
    compat.uninstall()
    cls = g["DoubleIntegratorCuda"]
    assert _compile(cls.__new__(cls)._dynamics_cuda_src(), 2) > 1000


def test_wrong_dimension_and_broken_source_are_compile_errors_with_the_log():
    lib = _ffi.lib()
    assert lib.pi_rollout_compile_check(_plugin_src("pendulum").encode(), 4, None) == _ffi.PI_ERR_COMPILE
    msg = lib.pi_last_error().decode()
    assert "PI_CALL_STEP_DYNAMICS" in msg and "error" in msg.lower()
    bad = "__device__ void step_dynamics(float a, float b, float u, float* x, float* y, float* r, bool* t) { oops; }"
    assert lib.pi_rollout_compile_check(bad.encode(), 2, None) == _ffi.PI_ERR_COMPILE
    msg = lib.pi_last_error().decode()
    assert "oops" in msg and "error" in msg.lower()
    assert lib.pi_rollout_compile_check(None, 2, None) == _ffi.PI_ERR_INVALID
    assert lib.pi_rollout_compile_check(b"", 7, None) == _ffi.PI_ERR_INVALID


def test_second_compile_is_a_disk_cache_hit(tmp_path, monkeypatch):
    lib = _ffi.lib()
    monkeypatch.setenv("DPB200_CACHE_DIR", str(tmp_path / "cache"))
    monkeypatch.delenv("DPB200_CACHE", raising=False)

    def counters():
        a, b = C.c_int64(), C.c_int64()
        lib.pi_nvrtc_counters(C.byref(a), C.byref(b))
        return a.value, b.value

    src = _plugin_src("cartpole")
    c0, h0 = counters()
    n1 = _compile(src, 4)
    assert counters() == (c0 + 1, h0)
    assert _compile(src, 4) == n1 and counters() == (c0 + 1, h0 + 1)
    # the table builder's entry for the same text is a different program
    n = C.c_int64()
    _ffi.check(lib.pi_compile_check(src.encode(), 4, C.byref(n)))
    assert counters() == (c0 + 2, h0 + 1) and len(list((tmp_path / "cache").glob("*.cubin"))) == 2


def test_rollout_without_a_device_fails_loudly():
    from dynamicprogramming_b200.utils import PolicyRollout

    if _ffi.lib().pi_device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(_ffi.EngineError) as ei:
        PolicyRollout(np.zeros(4, np.int32), np.ones(2, np.float32), [0, 0], [1, 1], [2, 2], _plugin_src("pendulum"))
    assert ei.value.code == _ffi.PI_ERR_NO_DEVICE
    assert "no CPU fallback" in str(ei.value)


def test_runner_parser_accepts_rollout_default_off():
    for name in runners.RUNNERS:
        assert not runners.build_parser(name).parse_args([]).rollout
        a = runners.build_parser(name).parse_args(["--rollout", "--episodes", "16", "--steps", "50"])
        assert a.rollout and (a.episodes, a.steps) == (16, 50)
