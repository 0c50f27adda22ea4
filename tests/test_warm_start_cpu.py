"""Warm start on a machine without a GPU: the C ABI entry point and its binding, the ahead-of-time prolongation kernel
in the sm_100a library, host-side validation of a warm-start source, and the runner's flags."""
import ctypes as C
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from dynamicprogramming_b200 import _ffi, envs, runners

ROOT = Path(__file__).resolve().parents[1]


def test_pi_prolong_values_is_exported_with_its_argtypes():
    assert "pi_prolong_values" in (ROOT / "include" / "dpb200.h").read_text()
    restype, argtypes = _ffi.SIGNATURES["pi_prolong_values"]
    assert restype is C.c_int
    assert argtypes == [C.c_void_p, C.POINTER(_ffi.PiGrid), C.c_void_p, C.POINTER(C.c_float)]
    fn = _ffi.lib().pi_prolong_values
    assert fn.argtypes == argtypes


def test_null_arguments_are_refused_without_a_device():
    lib = _ffi.lib()
    assert lib.pi_prolong_values(None, None, None, None) == _ffi.PI_ERR_INVALID
    assert "null" in lib.pi_last_error().decode()


def test_prolongation_kernel_is_in_the_sm_100a_library():
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not Path(cuobjdump).exists():
        pytest.skip("cuobjdump is not installed")
    out = subprocess.run([cuobjdump, "-symbols", str(Path(_ffi._LIB_PATH))], capture_output=True, text=True,
                         check=True).stdout
    assert "sm_100a" in subprocess.run([cuobjdump, "--list-elf", str(Path(_ffi._LIB_PATH))], capture_output=True,
                                       text=True, check=True).stdout
    for D in range(1, 7):
        assert f"_ZN2pi21prolong_values_kernelILi{D}E" in out, D


def _no_engine():
    """An engine object with no native engine behind it: anything that reached the device would fail."""
    cls = envs.REGISTRY["pendulum"].cls
    inst = cls.__new__(cls)
    inst._engine = None
    return inst


def test_warm_start_validates_the_value_count_before_the_device():
    vals = np.zeros(11, np.float32)
    with pytest.raises(_ffi.EngineError, match="11 values for a grid of shape \\[3, 4\\]"):
        _no_engine().warm_start((vals, [0, 0], [1, 1], [3, 4]))


def test_warm_start_validates_npz_keys_before_the_device(tmp_path):
    np.savez(tmp_path / "partial.npz", value_function=np.zeros(12, np.float32), bounds_low=np.zeros(2, np.float32),
             grid_shape=np.array([3, 4], np.int32))
    with pytest.raises(KeyError, match="bounds_high"):
        _no_engine().warm_start(tmp_path / "partial.npz")
    with pytest.raises(FileNotFoundError):
        _no_engine().warm_start(tmp_path / "missing.npz")


def test_runner_parser_takes_the_warm_start_flags():
    for name in runners.RUNNERS:
        p = runners.build_parser(name)
        a = p.parse_args([])
        assert a.warm_start_bins is None and a.warm_start_from is None
        b = p.parse_args(["--bins", "20", "--warm-start-bins", "12"])
        assert b.bins == 20 and b.warm_start_bins == 12 and b.warm_start_from is None
        c = p.parse_args(["--warm-start-from", "coarse.npz"])
        assert str(c.warm_start_from) == "coarse.npz" and c.warm_start_bins is None
        with pytest.raises(SystemExit):
            p.parse_args(["--warm-start-bins", "12", "--warm-start-from", "coarse.npz"])
    assert envs.REGISTRY["double_cartpole_swingup"].default_bins > 12
