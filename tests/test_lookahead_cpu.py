"""N8 one-step lookahead (include/dpb200.h: pi_rollout_lookahead / pi_rollout_run_lookahead) on a box without a GPU:
the rollout program, which now also holds the lookahead kernels, compiles for sm_100a against every plugin and for
D = 1..6, and the Python layer rejects bad arguments before any device call."""
import ctypes as C
import importlib.util
from pathlib import Path

import numpy as np
import pytest

from dynamicprogramming_b200 import _ffi, envs, runners
from dynamicprogramming_b200.utils import PolicyRollout

ROOT = Path(__file__).resolve().parents[1]
_spec = importlib.util.spec_from_file_location("odd_dims", ROOT / "tests" / "fixtures" / "odd_dims.py")
odd = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(odd)

KERNELS = (b"pi_rollout_episodes", b"pi_step_states", b"pi_lookahead_points", b"pi_rollout_lookahead")


def _plugin_src(name: str) -> str:
    spec = envs.REGISTRY[name]
    inst = spec.cls.__new__(spec.cls)
    for k, v in spec.kwargs.items():
        setattr(inst, k, v)
    return inst._dynamics_cuda_src()


def _compiled_cubin(src: str, D: int, tmp_path, monkeypatch) -> bytes:
    monkeypatch.setenv("DPB200_DUMP_JIT", str(tmp_path))
    n = C.c_int64()
    _ffi.check(_ffi.lib().pi_rollout_compile_check(src.encode(), D, C.byref(n)))
    cubin = (tmp_path / "pi_rollout.cu.cubin").read_bytes()
    assert len(cubin) == n.value
    return cubin


@pytest.mark.parametrize("name", sorted(envs.REGISTRY))
def test_lookahead_kernels_compile_for_every_plugin(name, tmp_path, monkeypatch):
    cubin = _compiled_cubin(_plugin_src(name), envs.REGISTRY[name].cls.N_DIMS, tmp_path, monkeypatch)
    for k in KERNELS:
        assert k in cubin, k


@pytest.mark.parametrize("D", [1, 2, 3, 4, 5, 6])
def test_lookahead_kernels_compile_for_every_dimension(D, tmp_path, monkeypatch):
    cubin = _compiled_cubin(odd.dynamics_src(D), D, tmp_path, monkeypatch)
    for k in KERNELS:
        assert k in cubin, k


def _no_device_rollout(D: int, n_states: int, n_actions: int) -> PolicyRollout:
    """A PolicyRollout whose handle must never be reached."""
    h = PolicyRollout.__new__(PolicyRollout)
    h.n_dims, h.n_states = D, n_states
    h.action_space = np.arange(n_actions, dtype=np.float32)
    h._h = None
    return h


def test_policy_rollout_validates_before_any_device_call():
    h = _no_device_rollout(2, 16, 3)
    with pytest.raises(ValueError, match="controller"):
        h.run(np.zeros((4, 2), np.float32), 5, 0.9, controller="greedy")
    with pytest.raises(ValueError, match="columns"):
        h.lookahead(np.zeros((4, 3), np.float32), 0.9)
    with pytest.raises(ValueError, match="16 states"):
        h.set_values(np.zeros(15, np.float32))


def test_engine_validates_before_any_device_call(monkeypatch):
    spec = envs.REGISTRY["cartpole"]
    eng = spec.cls.__new__(spec.cls)
    eng._engine = None

    def no_device(*args, **kwargs):
        raise AssertionError("a device call was made")

    monkeypatch.setattr(spec.cls, "_rollout_handle", no_device)
    D = spec.cls.N_DIMS
    with pytest.raises(ValueError, match="controller"):
        eng.rollout(np.zeros((3, D), np.float32), 5, gamma=0.9, controller="Lookahead")
    with pytest.raises(ValueError, match="columns"):
        eng.lookahead(np.zeros((3, D + 1), np.float32), gamma=0.9)


def test_lookahead_entry_points_reject_a_null_handle():
    lib = _ffi.lib()
    x = np.zeros((1, 2), np.float32)
    assert lib.pi_rollout_set_values(None, _ffi.ptr(x)) == _ffi.PI_ERR_INVALID
    assert lib.pi_rollout_lookahead(None, _ffi.ptr(x), 1, 0.9, None, None) == _ffi.PI_ERR_INVALID
    assert lib.pi_rollout_run_lookahead(None, _ffi.ptr(x), 1, 5, 0.9, None, None, None, None, None, None, None,
                                        None) == _ffi.PI_ERR_INVALID


def test_runner_parser_rollout_controller():
    for name in runners.RUNNERS:
        assert runners.build_parser(name).parse_args([]).rollout_controller == "policy"
        a = runners.build_parser(name).parse_args(["--rollout", "--rollout-controller", "lookahead"])
        assert a.rollout and a.rollout_controller == "lookahead"
    with pytest.raises(SystemExit):
        runners.build_parser("pendulum_cuda").parse_args(["--rollout-controller", "greedy"])


def test_format_rollout_names_only_a_non_default_controller():
    r = {"episodes": 2, "steps": 3, "mean_return": 1.0, "mean_discounted_return": 0.5, "mean_length": 3.0,
         "terminated": 0.0}
    assert runners.format_rollout(r).startswith("[=] rollout 2 episodes x 3 steps |")
    assert runners.format_rollout({**r, "controller": "lookahead"}).startswith(
        "[=] rollout (lookahead controller) 2 episodes x 3 steps |")
