"""SURVEY §8f N1: reference-style runner scripts run UNMODIFIED on the engine through
dynamicprogramming_b200.compat (sys.modules drop-ins for src.cuda_policy_iteration, and for cupy /
matplotlib only where they are missing)."""
import ctypes as C
import os
import sys
from pathlib import Path

import numpy as np
import pytest

from dynamicprogramming_b200 import _ffi, compat, engine

FIXTURE = Path(__file__).resolve().parent / "fixtures" / "double_integrator_cuda.py"
# a checkout of the original project (its runners/*_cuda.py); the test that loads them skips without one
REFERENCE = Path(os.environ["DPB200_REFERENCE"]) if os.environ.get("DPB200_REFERENCE") else None
REF_RUNNERS = {
    "pendulum_cuda": ("PendulumCuda", 2), "mountain_car_cuda": ("MountainCarCuda", 2),
    "continuous_mountain_car_cuda": ("ContinuousMountainCarCuda", 2), "cartpole_cuda": ("CartPoleCuda", 4),
    "cartpole_swingup_cuda": ("CartPoleSwingUpCuda", 4), "double_pendulum_swingup_cuda": ("DoublePendulumSwingUpCuda", 4),
    "overhead_crane_cuda": ("OverheadCraneCuda", 4), "double_cartpole_cuda": ("DoubleCartPoleCuda", 6),
    "double_cartpole_swingup_cuda": ("DoubleCartPoleSwingUpCuda", 6),
}
BASES = {2: engine.CudaPolicyIteration2D, 4: engine.CudaPolicyIteration4D, 6: engine.CudaPolicyIteration6D}


@pytest.fixture()
def installed():
    yield compat.install()
    compat.uninstall()


def _compiles(src: str, D: int) -> int:
    n = C.c_int64()
    _ffi.check(_ffi.lib().pi_compile_check(src.encode(), D, C.byref(n)))
    return n.value


def test_install_registers_the_engine_under_the_reference_module_name(installed):
    import src.cuda_policy_iteration as m   # noqa: the name the reference's runners import

    assert m.CudaPolicyIteration2D is engine.CudaPolicyIteration2D
    assert m.CudaPolicyIteration4D is engine.CudaPolicyIteration4D
    assert m.CudaPolicyIteration6D is engine.CudaPolicyIteration6D
    assert m.CudaPIConfig is engine.CudaPIConfig and m.GPU_AVAILABLE is True
    if installed["cupy_stub"]:
        import cupy as cp

        a = cp.asarray(np.array([1, 0, 1]), dtype=cp.bool_)
        assert a.dtype == np.bool_ and a.tolist() == [True, False, True]
        cp.get_default_memory_pool().free_all_blocks()
        with pytest.raises(AttributeError, match="cupy is not installed"):
            cp.RawModule
    if installed["matplotlib_stub"]:
        import matplotlib.pyplot as plt

        with pytest.raises(RuntimeError, match="--no-plot"):
            plt.figure()


def test_uninstall_removes_only_what_install_added():
    before = {k for k in sys.modules if k.split(".")[0] in ("src", "cupy", "matplotlib")}
    compat.install()
    compat.uninstall()
    after = {k for k in sys.modules if k.split(".")[0] in ("src", "cupy", "matplotlib")}
    assert after == before


def test_reference_style_fixture_runner_loads_unmodified(installed):
    g = compat.load_runner(FIXTURE)
    cls = g["DoubleIntegratorCuda"]
    assert issubclass(cls, engine.CudaPolicyIteration2D)
    assert list(g["BINS_SPACE"]) == ["pos", "vel"] and g["ACTION_SPACE"].dtype == np.float32
    inst = cls.__new__(cls)
    assert _compiles(inst._dynamics_cuda_src(), 2) > 0


@pytest.mark.skipif(REFERENCE is None, reason="DPB200_REFERENCE (a checkout of the original project) is not set")
@pytest.mark.parametrize("runner", sorted(REF_RUNNERS))
def test_every_reference_runner_imports_and_subclasses_the_engine(runner, installed):
    """The nine runners/*_cuda.py of the reference, executed as modules from where they lie: each one's
    `...Cuda` class becomes a subclass of the B200 engine and its dynamics string compiles through the
    engine's table-build kernel (NVRTC, sm_100a) — no GPU needed for either."""
    cls_name, D = REF_RUNNERS[runner]
    g = compat.load_runner(REFERENCE / "runners" / f"{runner}.py")
    cls = g[cls_name]
    assert issubclass(cls, BASES[D])
    assert len(g["BINS_SPACE"]) == D and callable(g["train"])
    inst = cls.__new__(cls)
    if runner == "overhead_crane_cuda":
        inst.target_x = -2.5
    assert _compiles(inst._dynamics_cuda_src(), D) > 0


# --------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_fixture_runner_trains_through_its_own_main_block(tmp_path, capsys):
    """`python double_integrator_cuda.py --bins 37 --retrain --no-plot --save-path ...` with the engine
    swapped in; the saved policy equals the same problem solved through the native plugin surface
    (explicit set_values instead of the cupy-mask store)."""
    save = tmp_path / "out" / "di_policy.npz"
    compat.run_runner(FIXTURE, ["--bins", "37", "--retrain", "--no-plot", "--save-path", str(save)])
    compat.uninstall()
    assert "states=1369" in capsys.readouterr().out
    got = np.load(save)
    assert set(got.files) == {"value_function", "policy", "bounds_low", "bounds_high", "grid_shape", "strides",
                              "corner_bits", "action_space", "states_space"}

    g = compat.load_runner(FIXTURE)
    compat.uninstall()
    base = g["DoubleIntegratorCuda"]

    class Native(base):
        def _allocate_tensors_and_compile(self):
            engine.CudaPolicyIteration2D._allocate_tensors_and_compile(self)
            self.set_values(self._goal_mask, 7.5)

    bins = {k: np.linspace(v[0], v[-1], 37, dtype=np.float32) for k, v in g["BINS_SPACE"].items()}
    pi = Native(bins, g["ACTION_SPACE"], engine.CudaPIConfig(gamma=0.97, theta=1e-4, max_eval_iter=2000, max_pi_iter=40))
    goal, states = pi._goal_mask.copy(), pi.states_space
    pi.run()
    np.testing.assert_array_equal(got["policy"], pi.policy)
    np.testing.assert_array_equal(got["value_function"].view(np.uint32), pi.value_function.view(np.uint32))
    # absorbing states keep their initial values: goal 7.5 (mask store), walls -50 (terminal value)
    assert goal.sum() > 0 and np.all(got["value_function"][goal] == 7.5)
    walls = (np.abs(states[:, 0]) >= 2.0)
    assert np.all(got["value_function"][walls & ~goal] == -50.0)
    assert got["value_function"][~walls & ~goal].max() < 7.5


@pytest.mark.gpu
def test_mask_store_hits_one_buffer_only():
    g = compat.load_runner(FIXTURE)
    compat.uninstall()
    cls = g["DoubleIntegratorCuda"]

    class Plain(cls):
        def _allocate_tensors_and_compile(self):
            engine.CudaPolicyIteration2D._allocate_tensors_and_compile(self)

    pi = Plain(g["BINS_SPACE"], g["ACTION_SPACE"])
    mask = np.zeros(pi.n_states, bool)
    mask[[3, 500, pi.n_states - 1]] = True
    pi.d_new_value_function[mask] = 2.25
    v, _ = pi.download()
    assert not np.any(v[mask] == 2.25)          # d_value_function untouched
    pi.d_value_function[mask] = 1.5
    v, _ = pi.download()
    assert np.all(v[mask] == 1.5) and np.all(v[~mask & ~pi._terminal_mask_host.astype(bool)] == 0.0)
    with pytest.raises(TypeError):
        pi.d_value_function[3] = 1.0
    with pytest.raises(TypeError):
        pi.d_policy[mask] = 1
    pi.close()
