"""Edge cases of the CUDA path: ragged grids, minimum sizes, sizes that are not
multiples of the block/warp, single action, all-terminal grids, error paths,
host<->device hand-off, the crane's goal initialisation."""
import numpy as np
import pytest
import torch

from dynamicprogramming_b200 import _ffi, envs
from dynamicprogramming_b200.engine import CudaPIConfig, CudaPolicyIteration2D, CudaPolicyIteration4D

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.mark.parametrize("env,shape", [("pendulum", (2, 2)), ("pendulum", (3, 257)), ("pendulum", (33, 7)),
                                       ("cartpole", (2, 3, 4, 5)), ("cartpole", (5, 2, 2, 9)),
                                       ("double_cartpole", (2, 2, 3, 2, 4, 3))])
def test_ragged_and_minimal_grids_match_the_reference(env, shape, reference):
    spec = envs.REGISTRY[env]
    cfg = spec.config()
    cfg.max_pi_iter, cfg.max_eval_iter = 3, 200
    names = list(spec.bounds)
    bins_space = {k: np.linspace(spec.bounds[k][0], spec.bounds[k][1], n, dtype=np.float32) for k, n in zip(names, shape)}
    eng = spec.cls(bins_space, spec.actions, cfg)
    assert eng.n_states == int(np.prod(shape))
    eng.run()
    reference.check_run(eng)


def test_single_action_and_fine_action_grid(reference):
    for actions in (np.array([0.5], np.float32), np.linspace(-1, 1, 201, dtype=np.float32)):
        spec = envs.REGISTRY["continuous_mountain_car"]
        cfg = spec.config()
        cfg.max_pi_iter = 2
        eng = spec.make(bins=40, actions=actions, config=cfg)
        eng.run()
        reference.check(f"{len(actions)} actions policy", eng.policy)
        reference.check(f"{len(actions)} actions value_function", eng.value_function)


class _AllTerminal(CudaPolicyIteration2D):
    def _dynamics_cuda_src(self):
        return ("__device__ void step_dynamics(float a, float b, float u, float* x, float* y, float* r, bool* t)"
                "{ *x = a; *y = b; *r = 1.0f; *t = false; }")

    def _terminal_fn(self, states):
        return np.ones(len(states), dtype=bool), 7.5


def test_all_states_terminal():
    bins = {"a": np.linspace(0, 1, 5, dtype=np.float32), "b": np.linspace(0, 1, 6, dtype=np.float32)}
    eng = _AllTerminal(bins, np.array([0.0, 1.0], np.float32), CudaPIConfig(max_pi_iter=3))
    eng.run()
    assert eng.pi_iterations == 1 and eng.total_eval_sweeps == 1      # delta = 0 at the first sync sweep
    np.testing.assert_array_equal(eng.value_function, np.float32(7.5))
    np.testing.assert_array_equal(eng.policy, 0)


class _Stay(CudaPolicyIteration2D):
    """Successor = the state itself, reward = action: V -> a_max / (1 - gamma), policy = argmax."""

    def _dynamics_cuda_src(self):
        return ("__device__ void step_dynamics(float a, float b, float u, float* x, float* y, float* r, bool* t)"
                "{ *x = a; *y = b; *r = u; *t = false; }")


def test_known_fixed_point_and_tie_break():
    bins = {"a": np.linspace(-1, 1, 9, dtype=np.float32), "b": np.linspace(-2, 2, 5, dtype=np.float32)}
    eng = _Stay(bins, np.array([0.25, 1.0, 1.0, -3.0], np.float32), CudaPIConfig(gamma=0.5, theta=1e-6, max_pi_iter=5))
    eng.run()
    np.testing.assert_array_equal(eng.policy, 1)                      # 1.0 appears twice: lowest index wins
    np.testing.assert_allclose(eng.value_function, 2.0, rtol=1e-5)


def test_nvrtc_error_surfaces_as_an_exception():
    class Broken(CudaPolicyIteration2D):
        def _dynamics_cuda_src(self):
            return "__device__ void step_dynamics(float a) { undeclared_symbol; }"

    bins = {"a": np.linspace(0, 1, 4, dtype=np.float32), "b": np.linspace(0, 1, 4, dtype=np.float32)}
    with pytest.raises(_ffi.EngineError) as ei:
        Broken(bins, np.array([0.0], np.float32))
    assert ei.value.code == _ffi.PI_ERR_COMPILE and "undeclared_symbol" in str(ei.value)


def test_call_order_and_argument_errors():
    eng = envs.make("pendulum", bins=8)
    lib = _ffi.lib()
    assert lib.pi_evaluate(eng._engine, None, None) == _ffi.PI_ERR_INVALID        # table not built yet
    eng.build_table()
    mask = np.zeros(eng.n_states, np.uint8)
    assert lib.pi_set_terminal(eng._engine, _ffi.ptr(mask), 0.0) == _ffi.PI_ERR_INVALID  # after the build
    assert lib.pi_expand_rows(eng._engine, 99, 0, 1, None, None, None, None) == _ffi.PI_ERR_INVALID
    assert lib.pi_expand_rows(eng._engine, 0, 0, eng.n_states + 1, None, None, None, None) == _ffi.PI_ERR_INVALID
    assert lib.pi_sweeps(eng._engine, 0, None, None) == _ffi.PI_ERR_INVALID
    assert b"n_sweeps" in lib.pi_last_error()
    eng.close()


def test_host_device_handoff_and_device_handles():
    eng = envs.make("cartpole", bins=6)
    N = eng.n_states
    rng = np.random.default_rng(0)
    V = rng.standard_normal(N).astype(np.float32)
    P = rng.integers(0, eng.n_actions, N).astype(np.int32)
    eng.upload_values(V)
    eng.upload_policy(P)
    v2, p2 = eng.download()
    np.testing.assert_array_equal(v2, V)
    np.testing.assert_array_equal(p2, P)
    t = torch.as_tensor(eng.d_value_function, device="cuda")          # zero-copy view through __cuda_array_interface__
    assert t.shape == (N,) and t.dtype == torch.float32
    # raw device handles are in the engine's storage order (pi_layout); host calls are in reference order
    np.testing.assert_array_equal(t.cpu().numpy(), eng.to_internal_order(V))
    np.testing.assert_array_equal(eng.d_policy.raw(), eng.to_internal_order(P))
    # .get() is what a reference-style subclass calls on its cupy arrays: reference order, whatever the storage order
    np.testing.assert_array_equal(eng.d_policy.get(), P)
    np.testing.assert_array_equal(eng.d_value_function.get(), V)
    lay = eng.layout()
    assert sorted(lay["perm"]) == list(range(4)) and lay["perm"][-1] == lay["fast_dim"]
    eng.close()


def test_crane_goal_states_start_at_one_over_one_minus_gamma(reference):
    spec = envs.REGISTRY["overhead_crane"]
    cfg = spec.config()
    cfg.max_pi_iter = 2
    eng = spec.make(bins=14, config=cfg)
    v0, _ = eng.download()
    goal = eng._goal_mask
    if goal.any():
        np.testing.assert_array_equal(v0[goal], np.float32(1.0 / (1.0 - cfg.gamma)))
    eng.run()
    reference.check("policy", eng.policy)
    reference.check("value_function", eng.value_function)


def test_max_eval_iter_cap_and_sync_schedule(reference):
    spec = envs.REGISTRY["pendulum"]
    for cap in (1, 7, 26, 40):
        cfg = spec.config()
        cfg.max_eval_iter, cfg.max_pi_iter = cap, 2
        eng = spec.make(bins=20, config=cfg)
        d_mine = eng.policy_evaluation()
        assert eng.last_eval_sweeps == cap
        reference.check_value(f"cap {cap} residual", float(np.float32(d_mine)))   # the residual the reference returns
        eng.close()


def test_saved_file_from_a_gpu_run(tmp_path):
    eng = envs.make("mountain_car", bins=30)
    eng.run()
    eng.save(tmp_path / "mc")
    d = np.load(tmp_path / "mc.npz")
    assert list(d.files) == ["value_function", "policy", "bounds_low", "bounds_high", "grid_shape", "strides",
                             "corner_bits", "action_space", "states_space"]
    assert d["policy"].dtype == np.int32 and d["value_function"].dtype == np.float32
    again = type(eng).load(tmp_path / "mc.npz")
    np.testing.assert_array_equal(again.policy, eng.policy)


@pytest.mark.parametrize("fast", ["ref", "0", "1", "auto"])
def test_storage_order_never_changes_results(fast, reference, monkeypatch):
    """Whatever dimension the engine stores contiguously, rows, V and policy stay bit-identical."""
    monkeypatch.setenv("DPB200_FAST_DIM", fast)
    spec = envs.REGISTRY["double_cartpole_swingup"]
    cfg = spec.config()
    cfg.max_pi_iter = 2
    eng = spec.make(bins=5, config=cfg)
    lay = eng.layout()
    if fast in ("0", "1"):
        assert lay["fast_dim"] == int(fast)
    if fast == "ref":
        assert lay["fast_dim"] == 5
    idx, w, r, t = eng.expand_rows(3)
    live = t == 0
    reference.check("action 3 idx", idx[live])
    reference.check("action 3 w", w[live])
    eng.run()
    reference.check_value("total_sweeps", eng.total_eval_sweeps)
    reference.check("policy", eng.policy)
    reference.check("value_function", eng.value_function)


def test_local_policy_upload_equals_the_full_upload():
    """pi_upload_policy_local (storage order, this rank's slice) == pi_upload_policy (reference order, whole grid)."""
    res = []
    rng = np.random.default_rng(3)
    P = None
    for local in (False, True):
        eng = envs.make("cartpole_swingup", bins=9)
        eng.build_table()
        if P is None:
            P = rng.integers(0, eng.n_actions, eng.n_states).astype(np.int32)
        if local:
            eng.upload_policy_local(eng.to_internal_order(P))
        else:
            eng.upload_policy(P)
        eng.sweeps(4)
        v, p = eng.download()
        res.append((bits(v).copy(), p.copy()))
        eng.close()
    np.testing.assert_array_equal(res[0][0], res[1][0])
    np.testing.assert_array_equal(res[0][1], res[1][1])
    np.testing.assert_array_equal(res[0][1], P)


@pytest.mark.parametrize("env,bins", [("pendulum", 64), ("mountain_car", 90), ("cartpole", 11), ("overhead_crane", 9)])
def test_persistent_multi_sweep_kernel_matches_the_reference(env, bins, monkeypatch, reference):
    """DPB200_PERSIST=on: one cooperative launch per sync interval (grid barrier between sweeps, rows in
    registers, L1-bypassing gathers) — same sweep counts, policy and V bits as the reference's kernels."""
    monkeypatch.setenv("DPB200_PERSIST", "on")
    monkeypatch.setenv("DPB200_XLINE", "off")
    spec = envs.REGISTRY[env]
    cfg = spec.config()
    cfg.max_pi_iter = 4
    eng = spec.make(bins=bins, config=cfg)
    eng.build_table()
    assert "eval_persistent_kernel" in eng.eval_kernel_info()["kernel"]
    eng.run()
    reference.check_run(eng)
