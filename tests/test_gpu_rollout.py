"""N5 closed-loop rollouts (include/dpb200.h: pi_rollout_*, csrc/rollout_src.cuh) on the device.

* The rollout's simulator is tied to the reference's kernels: one simulate_step per grid node and action reproduces
  the transition table (expand_rows, pinned bit for bit to the reference's kernels) in reward, termination and, through
  the host cell search of get_barycentric_Nd, in base index and weights.
* The fused kernel changes nothing: rollout() equals a Python loop of PolicyLookup + simulate_step bit for bit, and its
  returns equal host float64 sums in the defined order."""
from pathlib import Path

import numpy as np
import pytest

from dynamicprogramming_b200 import _ffi, compat, engine, envs, runners
from dynamicprogramming_b200.utils import PolicyLookup, PolicyRollout

pytestmark = pytest.mark.gpu

FIXTURE = Path(__file__).resolve().parent / "fixtures" / "double_integrator_cuda.py"
F32 = np.float32


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32 if np.asarray(a).dtype == np.float32 else np.uint64)


def _fixture_engine(max_pi_iter=2, max_eval_iter=60):
    g = compat.load_runner(FIXTURE)
    compat.uninstall()

    class Plain(g["DoubleIntegratorCuda"]):
        def _allocate_tensors_and_compile(self):
            engine.CudaPolicyIteration2D._allocate_tensors_and_compile(self)

    return Plain(g["BINS_SPACE"], g["ACTION_SPACE"],
                 engine.CudaPIConfig(gamma=0.97, max_pi_iter=max_pi_iter, max_eval_iter=max_eval_iter))


def _engine(env, bins, max_pi_iter=2, max_eval_iter=60):
    if env == "fixture":
        return _fixture_engine(max_pi_iter, max_eval_iter)
    spec = envs.REGISTRY[env]
    cfg = spec.config()
    cfg.max_pi_iter, cfg.max_eval_iter = max_pi_iter, max_eval_iter
    return spec.make(bins=bins, config=cfg)


def _cell_search(nx, lo, hi, shape):
    """get_barycentric_Nd as the table builder computes it, contraction-free, in float32 on the host:
    n = (x - lo) / (hi - lo) * (shape - 1); clamp to [0, shape-1]; i = min(trunc(n), shape - 2); f = n - i."""
    n, D = nx.shape
    idx = np.empty((n, D), np.int64)
    fr = np.empty((n, D), F32)
    for d in range(D):
        pn = ((nx[:, d] - F32(lo[d])).astype(F32) / F32(F32(hi[d]) - F32(lo[d]))).astype(F32)
        pn = (pn * F32(shape[d] - 1)).astype(F32)
        pn = np.maximum(F32(0), np.minimum(pn, F32(shape[d] - 1)))
        i = np.minimum(pn.astype(np.int64), shape[d] - 2)
        idx[:, d] = i
        fr[:, d] = (pn - i.astype(F32)).astype(F32)
    return idx, fr


def _corner_bit(D, c, d):
    return (c >> (1 - d)) & 1 if D == 2 else (c >> d) & 1


@pytest.mark.parametrize("env,bins", [("pendulum", 31), ("mountain_car", 31), ("continuous_mountain_car", 31),
                                      ("cartpole", 9), ("cartpole_swingup", 9), ("double_pendulum_swingup", 9),
                                      ("overhead_crane", 9), ("double_cartpole", 6), ("double_cartpole_swingup", 6),
                                      ("fixture", None)])
def test_simulate_step_reproduces_the_transition_table(env, bins):
    eng = _engine(env, bins)
    eng.build_table()
    D, shape = eng.N_DIMS, [int(s) for s in eng.grid_shape]
    stride = np.array(eng.strides, np.int64)
    states = eng.states_space
    C = 1 << D
    for a in range(eng.n_actions):
        idx, w, r, t = eng.expand_rows(a)
        live = t != 2                                  # absorbing rows (terminal mask) have no successor
        nx, rr, tt = eng.simulate_step(states[live], np.full(int(live.sum()), eng.action_space[a], F32))
        np.testing.assert_array_equal(bits(rr), bits(r[live]), err_msg=f"{env} action {a}: reward")
        np.testing.assert_array_equal(tt, t[live] == 1, err_msg=f"{env} action {a}: terminated")
        go = ~tt
        cell, fr = _cell_search(nx[go], eng.bounds_low, eng.bounds_high, shape)
        base = (cell * stride).sum(axis=1)
        idx_l, w_l = idx[live][go], w[live][go]
        for c in range(C):
            off = sum(_corner_bit(D, c, d) * int(stride[d]) for d in range(D))
            np.testing.assert_array_equal(idx_l[:, c], base + off, err_msg=f"{env} action {a} corner {c}: index")
            wc = np.ones(len(fr), F32)
            for d in range(D):
                wc = (wc * (fr[:, d] if _corner_bit(D, c, d) else (F32(1) - fr[:, d]).astype(F32))).astype(F32)
            np.testing.assert_array_equal(bits(wc), bits(w_l[:, c]), err_msg=f"{env} action {a} corner {c}: weight")
    eng.close()


def _loop_reference(eng, policy, x0, T, gamma):
    """The same episodes as a Python loop of PolicyLookup + simulate_step (two calls per step), and the returns as
    host float64 sums: total += r; ret += disc * r; disc *= gamma."""
    look = PolicyLookup(policy, eng.action_space, eng.bounds_low, eng.bounds_high, eng.grid_shape)
    n, D = x0.shape
    S = np.full((n, T + 1, D), np.nan, F32)
    A = np.full((n, T), np.nan, F32)
    R = np.full((n, T), np.nan, F32)
    S[:, 0] = x0
    x = x0.copy()
    length = np.zeros(n, np.int32)
    term = np.zeros(n, bool)
    for t in range(T):
        alive = np.nonzero(~term)[0]
        if len(alive) == 0:
            break
        a = look(x[alive])
        nx, r, tm = eng.simulate_step(x[alive], a)
        A[alive, t], R[alive, t], S[alive, t + 1] = a, r, nx
        x[alive] = nx
        length[alive] = t + 1
        term[alive] = tm
    look.close()
    total = np.zeros(n, np.float64)
    ret = np.zeros(n, np.float64)
    disc = np.ones(n, np.float64)
    for t in range(T):
        m = t < length
        r = R[m, t].astype(np.float64)
        total[m] = total[m] + r
        ret[m] = ret[m] + disc[m] * r
        disc[m] = disc[m] * np.float64(gamma)
    return dict(states=S, actions=A, rewards=R, length=length, terminated=term, final=x, total=total, ret=ret)


def _starts(eng, n, seed):
    rng = np.random.default_rng(seed)
    lo, hi = eng.bounds_low, eng.bounds_high
    return (lo + (hi - lo) * rng.uniform(-0.1, 1.1, (n, eng.N_DIMS))).astype(F32)   # includes out-of-grid starts


@pytest.mark.parametrize("env,bins,T,terminates", [("pendulum", 31, 150, False), ("cartpole", 9, 120, True),
                                                   ("mountain_car", 31, 150, True), ("double_cartpole_swingup", 6, 60, None),
                                                   ("fixture", None, 100, True)])
def test_fused_rollout_equals_lookup_plus_step_loop(env, bins, T, terminates):
    eng = _engine(env, bins, max_pi_iter=1)
    eng.policy_evaluation()
    eng.policy_improvement()            # the policy after one improvement
    _, policy = eng.download()
    x0 = _starts(eng, 700, 3)
    gamma = float(F32(eng.config.gamma))
    got = eng.rollout(x0, T, record=True)
    exp = _loop_reference(eng, policy, x0, T, gamma)
    np.testing.assert_array_equal(got.length, exp["length"])
    np.testing.assert_array_equal(got.terminated, exp["terminated"])
    np.testing.assert_array_equal(bits(got.states), bits(exp["states"]))     # incl. the NaN padding, bit for bit
    np.testing.assert_array_equal(bits(got.actions), bits(exp["actions"]))
    np.testing.assert_array_equal(bits(got.rewards), bits(exp["rewards"]))
    np.testing.assert_array_equal(bits(got.final_states), bits(exp["final"]))
    np.testing.assert_array_equal(bits(got.total_reward), bits(exp["total"]))
    np.testing.assert_array_equal(bits(got.discounted_return), bits(exp["ret"]))
    if terminates is False:
        assert not got.terminated.any() and np.all(got.length == T)
    elif terminates:
        assert got.terminated.any() and got.length.min() < T
    # record=False: the same summary outputs, bit for bit
    plain = eng.rollout(x0, T)
    assert plain.states is None and plain.actions is None and plain.rewards is None
    for name in ("total_reward", "discounted_return", "final_states"):
        np.testing.assert_array_equal(bits(getattr(plain, name)), bits(getattr(got, name)))
    np.testing.assert_array_equal(plain.length, got.length)
    np.testing.assert_array_equal(plain.terminated, got.terminated)
    eng.close()


def test_rollout_after_run_equals_rollout_after_load(tmp_path):
    spec = envs.REGISTRY["cartpole"]
    eng = spec.make(bins=8)
    eng.run()
    x0 = _starts(eng, 300, 5)
    a = eng.rollout(x0, 80, record=True)
    eng.save(tmp_path / "p")
    loaded = spec.cls.load(tmp_path / "p.npz")
    b = loaded.rollout(x0, 80, gamma=float(F32(spec.config().gamma)), record=True)
    for name in ("total_reward", "discounted_return", "final_states", "states", "actions", "rewards"):
        np.testing.assert_array_equal(bits(getattr(a, name)), bits(getattr(b, name)))
    np.testing.assert_array_equal(a.length, b.length)
    # a new policy object rebuilds the cached handle
    loaded.policy = np.zeros_like(loaded.policy)
    c = loaded.rollout(x0, 80, gamma=float(F32(spec.config().gamma)))
    assert not np.array_equal(c.total_reward, b.total_reward)


def test_edge_cases():
    eng = _engine("cartpole", 8, max_pi_iter=1)
    eng.policy_evaluation()
    eng.policy_improvement()
    D = eng.N_DIMS
    x0 = _starts(eng, 64, 9)
    # n_steps = 0: nothing happens
    z = eng.rollout(x0, 0, record=True)
    assert np.all(z.length == 0) and not z.terminated.any() and np.all(z.total_reward == 0.0)
    np.testing.assert_array_equal(bits(z.final_states), bits(x0))
    assert z.states.shape == (64, 1, D) and z.actions.shape == (64, 0)
    np.testing.assert_array_equal(bits(z.states[:, 0]), bits(x0))
    # zero episodes
    e = eng.rollout(np.zeros((0, D), F32), 10, record=True)
    assert e.length.shape == (0,) and e.states.shape == (0, 11, D)
    # a start whose first step terminates: length 1
    _, policy = eng.download()
    look = PolicyLookup(policy, eng.action_space, eng.bounds_low, eng.bounds_high, eng.grid_shape)
    cand = x0.copy()
    cand[:, 0] = np.where(np.arange(64) % 2, eng.bounds_high[0], eng.bounds_low[0]) * F32(1.5)
    _, _, tm = eng.simulate_step(cand, look(cand))
    look.close()
    assert tm.any()
    first = cand[np.nonzero(tm)[0][:1]]
    one = eng.rollout(first, 50, record=True)
    assert one.length[0] == 1 and one.terminated[0]
    assert np.isnan(one.actions[0, 1:]).all() and np.isnan(one.states[0, 2:]).all()
    # argument errors
    with pytest.raises(ValueError):
        eng.rollout(np.zeros((3, D + 1), F32), 5)
    with pytest.raises(ValueError):
        eng.simulate_step(np.zeros((3, D - 1), F32), np.zeros(3, F32))
    with pytest.raises(_ffi.EngineError) as ei:
        eng.rollout(x0, -1)
    assert ei.value.code == _ffi.PI_ERR_INVALID
    src = eng._dynamics_cuda_src()
    with pytest.raises(_ffi.EngineError) as ei:
        PolicyRollout(np.full(eng.n_states, eng.n_actions, np.int32), eng.action_space, eng.bounds_low, eng.bounds_high,
                      eng.grid_shape, src)
    assert ei.value.code == _ffi.PI_ERR_INVALID
    eng.close()


def test_runner_rollout_summary_equals_pi_rollout(tmp_path, capsys):
    path = tmp_path / "cartpole_cuda_policy.npz"
    assert runners.main(["cartpole_cuda", "--bins", "8", "--save-path", str(path), "--no-plot", "--rollout",
                         "--episodes", "16", "--steps", "50"]) == 0
    out = capsys.readouterr().out
    line = [ln for ln in out.splitlines() if ln.startswith("[=] rollout")]
    assert len(line) == 1
    spec = envs.REGISTRY["cartpole"]
    pi = spec.cls.load(path)
    res = pi.rollout(runners.start_states(pi, 16, 42), 50, gamma=float(F32(spec.config().gamma)))
    expect = runners.format_rollout({"episodes": 16, "steps": 50, "mean_return": float(res.total_reward.mean()),
                                     "mean_discounted_return": float(res.discounted_return.mean()),
                                     "mean_length": float(res.length.mean()), "terminated": float(res.terminated.mean())})
    assert line[0] == expect
    # without the flag the output has no rollout line
    assert runners.main(["cartpole_cuda", "--bins", "8", "--save-path", str(path), "--episodes", "2"]) == 0
    assert "[=] rollout" not in capsys.readouterr().out
