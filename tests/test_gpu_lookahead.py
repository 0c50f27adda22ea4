"""N8 one-step lookahead on a value table (include/dpb200.h: pi_rollout_set_values / pi_rollout_lookahead /
pi_rollout_run_lookahead, csrc/lookahead_src.cuh) on the device.

* At grid nodes the lookahead is the improvement pass: with the V that policy_improvement() reads, its winner is the
  action pi_improve writes at every non-absorbing node, in both table modes and in both storage orders.
* At arbitrary points its Q matrix equals, bit for bit, a host restatement: simulate_step (pinned to the transition table
  by tests/test_gpu_rollout.py), the builder's cell search without contraction, the improvement's corner order, and an
  exactly rounded fmaf.
* rollout(controller="lookahead") equals a Python loop of lookahead + simulate_step bit for bit."""
import importlib.util
from pathlib import Path

import numpy as np
import pytest

from dynamicprogramming_b200 import _ffi, envs, runners
from dynamicprogramming_b200.engine import CudaPIConfig, _CudaPolicyIterationBase
from dynamicprogramming_b200.utils import PolicyRollout

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
_spec = importlib.util.spec_from_file_location("odd_dims", ROOT / "tests" / "fixtures" / "odd_dims.py")
odd = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(odd)

F32 = np.float32
MODES = ("full", "recompute")
LAYOUTS = ("ref", "auto")
ENV_BINS = {"pendulum": 41, "mountain_car": 41, "continuous_mountain_car": 41, "cartpole": 9, "cartpole_swingup": 9,
            "double_pendulum_swingup": 9, "overhead_crane": 9, "double_cartpole": 5, "double_cartpole_swingup": 5}


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def assert_same_floats(got, want, what):
    """Bit-equal, except that any NaN matches any NaN (the device's NaN is the canonical one, the host keeps payloads)."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, what
    nan = np.isnan(got)
    np.testing.assert_array_equal(nan, np.isnan(want), err_msg=f"{what}: NaN positions")
    np.testing.assert_array_equal(bits(np.where(nan, 0, got).astype(got.dtype)),
                                  bits(np.where(nan, 0, want).astype(want.dtype)), err_msg=what)


def _set_env(monkeypatch, mode, layout):
    monkeypatch.setenv("DPB200_TABLE", mode)
    if layout == "auto":
        monkeypatch.delenv("DPB200_FAST_DIM", raising=False)
    else:
        monkeypatch.setenv("DPB200_FAST_DIM", layout)


def _adversarial_values(N, seed):
    rng = np.random.default_rng(seed)
    V = (rng.choice([-1.0, 1.0], N) * 10.0 ** rng.uniform(-12, 12, N)).astype(F32)
    V[rng.random(N) < 0.05] = F32(0.0)
    V[rng.random(N) < 0.05] = F32(-0.0)
    return V


def _improve_once(eng, V, P0):
    eng.upload_values(V)
    eng.upload_policy(P0)
    eng.policy_improvement()
    return eng.download()[1]


def _absorbing(eng):
    return eng._terminal_mask_and_value()[0]


# ── host restatement ───────────────────────────────────────────────────────────────────────────────────────────────

def fmaf(a, b, c):
    """Exactly rounded float32 fmaf: the float64 product of two float32 values is exact; the float64 sum is made
    round-to-odd with TwoSum, so rounding it to float32 is the correctly rounded a * b + c."""
    with np.errstate(all="ignore"):
        p = np.asarray(a, F32).astype(np.float64) * np.asarray(b, F32).astype(np.float64)
        c = np.asarray(c, F32).astype(np.float64)
        s = p + c
        bb = s - p
        err = (p - (s - bb)) + (c - bb)
        s = np.asarray(s, np.float64).copy()
        fix = np.isfinite(s) & (err != 0) & ((s.view(np.uint64) & 1) == 0)
        s[fix] = np.nextafter(s[fix], np.where(err[fix] > 0, np.inf, -np.inf))
        return s.astype(F32)


def cell_search(nx, lo, hi, shape):
    """pi_row's cell search in float32, contraction-free, with fminf / fmaxf semantics (a NaN successor lands where
    the device puts it)."""
    n, D = nx.shape
    idx = np.empty((n, D), np.int64)
    fr = np.empty((n, D), F32)
    with np.errstate(all="ignore"):
        for d in range(D):
            top = F32(shape[d] - 1)
            pn = ((nx[:, d] - F32(lo[d])).astype(F32) / F32(F32(hi[d]) - F32(lo[d]))).astype(F32)
            pn = (pn * top).astype(F32)
            pn = np.fmax(F32(0), np.fmin(pn, top))
            i = np.minimum(pn.astype(np.int64), shape[d] - 2)
            idx[:, d] = i
            fr[:, d] = (pn - i.astype(F32)).astype(F32)
    return idx, fr


def _corner_bit(D, c, d):
    return (c >> (1 - d)) & 1 if D == 2 else (c >> d) & 1


def host_q(eng, V, points, gamma):
    """Q (n, A) of the lookahead's definition on the host (V in reference order)."""
    D, shape = eng.N_DIMS, [int(s) for s in eng.grid_shape]
    stride = np.array(eng.strides, np.int64)
    n, A = len(points), len(eng.action_space)
    Q = np.empty((n, A), F32)
    for a in range(A):
        nx, r, term = eng.simulate_step(points, np.full(n, eng.action_space[a], F32))
        ev = np.zeros(n, F32)
        go = ~term
        cell, fr = cell_search(nx[go], eng.bounds_low, eng.bounds_high, shape)
        base = (cell * stride).sum(axis=1)
        e = np.zeros(int(go.sum()), F32)
        for c in range(1 << D):
            off = sum(_corner_bit(D, c, d) * int(stride[d]) for d in range(D))
            w = np.ones(len(fr), F32)
            for d in range(D):
                w = (w * (fr[:, d] if _corner_bit(D, c, d) else (F32(1) - fr[:, d]).astype(F32))).astype(F32)
            e = fmaf(w, V[base + off], e)
        ev[go] = e
        Q[:, a] = fmaf(np.full(n, gamma, F32), ev, r)
    return Q


def host_winner(Q):
    best = np.zeros(len(Q), np.int32)
    best_q = np.full(len(Q), F32(-1e30), F32)
    for a in range(Q.shape[1]):
        win = Q[:, a] > best_q               # NaN never wins, ties keep the lower index
        best[win] = a
        best_q[win] = Q[win, a]
    return best


# ── 1. nodes equal the improvement pass ────────────────────────────────────────────────────────────────────────────

def _check_nodes(eng, seed):
    N = eng.n_states
    V = _adversarial_values(N, seed)
    P0 = np.random.default_rng(seed + 1).integers(0, eng.n_actions, N).astype(np.int32)
    P1 = _improve_once(eng, V, P0)
    idx, act = eng.lookahead(eng.states_space)
    live = ~_absorbing(eng)
    assert live.any()
    np.testing.assert_array_equal(idx[live], P1[live])
    np.testing.assert_array_equal(bits(act), bits(eng.action_space.astype(F32)[idx]))


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", sorted(ENV_BINS))
def test_lookahead_at_nodes_equals_the_improvement_for_every_environment(name, mode, layout, monkeypatch):
    _set_env(monkeypatch, mode, layout)
    spec = envs.REGISTRY[name]
    eng = envs.make(name, bins=ENV_BINS[name], config=spec.config())
    eng.build_table()
    assert eng.engine_stats()["table_mode"] == mode
    _check_nodes(eng, 500 + sorted(ENV_BINS).index(name))
    eng.close()


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("D", [1, 3, 5])
def test_lookahead_at_nodes_equals_the_improvement_for_the_odd_dims_fixture(D, mode, layout, monkeypatch):
    _set_env(monkeypatch, mode, layout)
    eng = odd.make(D)
    eng.build_table()
    assert eng.engine_stats()["table_mode"] == mode
    _check_nodes(eng, 600 + D)
    eng.close()


# ── 2. edge rewards ────────────────────────────────────────────────────────────────────────────────────────────────

class EdgeRewards(_CudaPolicyIterationBase):
    """Every state stays where it is; the reward depends on the action and on the state's class ix % 4:
    0: NaN, -inf, -1e30, -0, +0, +0, 1, -0   (action 6 wins)
    1: NaN, -inf, -1e30, NaN, -2e30, NaN, -inf, -1e30   (nothing competes: action 0)
    2: NaN, -inf, -1e30, -0, +0, +0, -0, +0   (signed zeros and exact ties)
    3: -9.9e29, -1e30, NaN, 2, 2, +inf, 2, NaN   (+inf wins)"""
    N_DIMS = 2

    def _dynamics_cuda_src(self) -> str:
        return r"""
__device__ void step_dynamics(float x, float y, float u, float* nx, float* ny, float* reward, bool* terminated)
{
    const float nan = __int_as_float(0x7fc00000), inf = __int_as_float(0x7f800000);
    const float tab[4][8] = {
        {nan, -inf, -1e30f, -0.0f, 0.0f, 0.0f, 1.0f, -0.0f},
        {nan, -inf, -1e30f, nan, -2e30f, nan, -inf, -1e30f},
        {nan, -inf, -1e30f, -0.0f, 0.0f, 0.0f, -0.0f, 0.0f},
        {-9.9e29f, -1e30f, nan, 2.0f, 2.0f, inf, 2.0f, nan}};
    *nx = x;
    *ny = y;
    *reward = tab[((int)(x + 0.5f)) & 3][(int)u];
    *terminated = false;
}
"""


@pytest.mark.parametrize("mode", MODES)
def test_nan_inf_signed_zero_and_tied_rewards_pick_the_improvements_winner(mode, monkeypatch):
    _set_env(monkeypatch, mode, "auto")
    space = {"x": np.arange(16, dtype=F32), "y": np.linspace(-1, 1, 9, dtype=F32)}
    acts = np.arange(8, dtype=F32)
    rng = np.random.default_rng(5)
    eng = EdgeRewards(space, acts, CudaPIConfig(gamma=0.5))
    N = eng.n_states
    cls = (np.arange(16)[:, None] & 3).repeat(9, axis=1).ravel()
    for V in (np.zeros(N, F32), np.full(N, -1.4e-45, F32),
              rng.choice(np.array([0.0, -0.0, -1.4e-45, 1.4e-45, 1e-40, -1e-40, 5.0, -5.0], F32), N)):
        P1 = _improve_once(eng, V.astype(F32), rng.integers(0, 8, N).astype(np.int32))
        idx, _, q = eng.lookahead(eng.states_space, q=True)
        np.testing.assert_array_equal(idx, P1)
        np.testing.assert_array_equal(idx, host_winner(q))
        assert (idx[cls == 0] == 6).all() and (idx[cls == 1] == 0).all() and (idx[cls == 3] == 5).all()
        assert_same_floats(q, host_q(eng, V.astype(F32), eng.states_space, F32(0.5)), "Q")
    eng.close()


# ── 3. arbitrary points, exact Q ───────────────────────────────────────────────────────────────────────────────────

def _points(eng, n, seed):
    rng = np.random.default_rng(seed)
    lo, hi = eng.bounds_low.astype(np.float64), eng.bounds_high.astype(np.float64)
    p = (lo + (hi - lo) * rng.uniform(-0.2, 1.2, (n, eng.N_DIMS))).astype(F32)   # includes out-of-grid points
    specials = np.array([np.nan, np.inf, -np.inf], F32)
    for k in range(min(3 * eng.N_DIMS, n)):
        p[k, k % eng.N_DIMS] = specials[k % 3]
    return p


@pytest.mark.parametrize("name", ["pendulum", "mountain_car", "cartpole", "double_pendulum_swingup",
                                  "double_cartpole_swingup", "odd3", "odd5"])
def test_q_at_arbitrary_points_equals_the_host_restatement(name, monkeypatch):
    monkeypatch.delenv("DPB200_FAST_DIM", raising=False)
    monkeypatch.delenv("DPB200_TABLE", raising=False)
    if name.startswith("odd"):
        eng = odd.make(int(name[3:]))
    else:
        eng = envs.make(name, bins=ENV_BINS[name], config=envs.REGISTRY[name].config())
    V = _adversarial_values(eng.n_states, 77)
    V[::97] = F32(np.nan)
    eng.upload_values(V)
    V = eng.download()[0]               # what the engine holds (absorbing states keep their terminal value)
    pts = _points(eng, 3000, 8)
    gamma = F32(eng.config.gamma)
    idx, act, q = eng.lookahead(pts, q=True)
    Q = host_q(eng, V, pts, gamma)
    assert_same_floats(q, Q, f"{name}: Q")
    np.testing.assert_array_equal(idx, host_winner(Q))
    np.testing.assert_array_equal(bits(act), bits(eng.action_space.astype(F32)[idx]))
    # without q: the same indices; another gamma: the same host rule
    idx2, _ = eng.lookahead(pts)
    np.testing.assert_array_equal(idx2, idx)
    idx3, _, q3 = eng.lookahead(pts, gamma=0.25, q=True)
    assert_same_floats(q3, host_q(eng, V, pts, F32(0.25)), f"{name}: Q at gamma 0.25")
    np.testing.assert_array_equal(idx3, host_winner(q3))
    eng.close()


# ── 4. a stable policy is its own lookahead ─────────────────────────────────────────────────────────────────────────

@pytest.mark.parametrize("name,bins", [("cartpole", 8), ("pendulum", 31)])
def test_lookahead_at_nodes_equals_a_stable_policy(name, bins):
    eng = envs.make(name, bins=bins)
    eng.run()
    assert eng.converged
    idx, _ = eng.lookahead(eng.states_space)        # host value_function after run()
    live = ~_absorbing(eng)
    np.testing.assert_array_equal(idx[live], eng.policy[live])


# ── 5. rollouts ────────────────────────────────────────────────────────────────────────────────────────────────────

def _loop_reference(eng, choose, x0, T, gamma):
    """Episodes as a Python loop of choose(x) + simulate_step, returns as host float64 sums."""
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
        a = choose(x[alive])
        nx, r, tm = eng.simulate_step(x[alive], a)
        A[alive, t], R[alive, t], S[alive, t + 1] = a, r, nx
        x[alive] = nx
        length[alive] = t + 1
        term[alive] = tm
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
    return (lo + (hi - lo) * rng.uniform(-0.1, 1.1, (n, eng.N_DIMS))).astype(F32)


def _assert_rollout(got, exp):
    np.testing.assert_array_equal(got.length, exp["length"])
    np.testing.assert_array_equal(got.terminated, exp["terminated"])
    np.testing.assert_array_equal(bits(got.states), bits(exp["states"]))
    np.testing.assert_array_equal(bits(got.actions), bits(exp["actions"]))
    np.testing.assert_array_equal(bits(got.rewards), bits(exp["rewards"]))
    np.testing.assert_array_equal(bits(got.final_states), bits(exp["final"]))
    np.testing.assert_array_equal(bits(got.total_reward), bits(exp["total"]))
    np.testing.assert_array_equal(bits(got.discounted_return), bits(exp["ret"]))


@pytest.mark.parametrize("name,bins,T", [("pendulum", 31, 150), ("cartpole", 9, 120), ("mountain_car", 31, 150),
                                         ("double_cartpole_swingup", 6, 60), ("odd3", None, 80)])
def test_lookahead_rollout_equals_lookahead_plus_step_loop(name, bins, T):
    if name.startswith("odd"):
        eng = odd.make(int(name[3:]), config=CudaPIConfig(gamma=odd.GAMMA, max_eval_iter=60, max_pi_iter=1))
    else:
        cfg = envs.REGISTRY[name].config()
        cfg.max_pi_iter, cfg.max_eval_iter = 1, 60
        eng = envs.make(name, bins=bins, config=cfg)
    eng.policy_evaluation()
    eng.policy_improvement()
    eng.policy_evaluation()            # V no longer the one the policy is greedy for
    x0 = _starts(eng, 700, 3)
    gamma = float(F32(eng.config.gamma))
    got = eng.rollout(x0, T, record=True, controller="lookahead")
    exp = _loop_reference(eng, lambda x: eng.lookahead(x)[1], x0, T, gamma)
    _assert_rollout(got, exp)
    plain = eng.rollout(x0, T, controller="lookahead")
    assert plain.states is None and plain.actions is None and plain.rewards is None
    for field in ("total_reward", "discounted_return", "final_states"):
        np.testing.assert_array_equal(bits(getattr(plain, field)), bits(getattr(got, field)))
    np.testing.assert_array_equal(plain.length, got.length)
    np.testing.assert_array_equal(plain.terminated, got.terminated)
    # the default controller is the interpolated grid policy, unchanged
    from dynamicprogramming_b200.utils import PolicyLookup
    _, policy = eng.download()
    look = PolicyLookup(policy, eng.action_space, eng.bounds_low, eng.bounds_high, eng.grid_shape)
    _assert_rollout(eng.rollout(x0, T, record=True), _loop_reference(eng, look, x0, T, gamma))
    look.close()
    # new values on the live engine reach the cached handle
    eng.upload_values(np.zeros(eng.n_states, F32))
    z = eng.rollout(x0, T, record=True, controller="lookahead")
    _assert_rollout(z, _loop_reference(eng, lambda x: eng.lookahead(x)[1], x0, T, gamma))
    eng.close()


def test_lookahead_rollout_after_run_equals_rollout_after_load(tmp_path):
    spec = envs.REGISTRY["cartpole"]
    eng = spec.make(bins=8)
    eng.run()
    x0 = _starts(eng, 300, 5)
    gamma = float(F32(spec.config().gamma))
    a = eng.rollout(x0, 80, record=True, controller="lookahead")
    la = eng.lookahead(x0, q=True)
    eng.save(tmp_path / "p")
    loaded = spec.cls.load(tmp_path / "p.npz")
    b = loaded.rollout(x0, 80, gamma=gamma, record=True, controller="lookahead")
    lb = loaded.lookahead(x0, gamma=gamma, q=True)
    for field in ("total_reward", "discounted_return", "final_states", "states", "actions", "rewards"):
        np.testing.assert_array_equal(bits(getattr(a, field)), bits(getattr(b, field)))
    np.testing.assert_array_equal(a.length, b.length)
    for u, v in zip(la, lb):
        np.testing.assert_array_equal(bits(u) if u.dtype == F32 else u, bits(v) if v.dtype == F32 else v)
    # a new value_function object is uploaded again
    loaded.value_function = np.zeros_like(loaded.value_function)
    _, _, q0 = loaded.lookahead(x0, gamma=gamma, q=True)
    assert not np.array_equal(q0, lb[2])


# ── 6. edge cases ──────────────────────────────────────────────────────────────────────────────────────────────────

def test_edge_cases():
    cfg = envs.REGISTRY["cartpole"].config()
    cfg.max_pi_iter, cfg.max_eval_iter = 1, 60
    eng = envs.make("cartpole", bins=8, config=cfg)
    eng.policy_evaluation()
    eng.policy_improvement()
    D, A = eng.N_DIMS, eng.n_actions
    x0 = _starts(eng, 64, 9)
    # n = 0
    idx, act, q = eng.lookahead(np.zeros((0, D), F32), q=True)
    assert idx.shape == (0,) and act.shape == (0,) and q.shape == (0, A)
    e = eng.rollout(np.zeros((0, D), F32), 10, record=True, controller="lookahead")
    assert e.length.shape == (0,) and e.states.shape == (0, 11, D)
    # n_steps = 0 and n_steps < 0
    z = eng.rollout(x0, 0, record=True, controller="lookahead")
    assert np.all(z.length == 0) and not z.terminated.any() and np.all(z.total_reward == 0.0)
    np.testing.assert_array_equal(bits(z.final_states), bits(x0))
    with pytest.raises(_ffi.EngineError) as ei:
        eng.rollout(x0, -1, controller="lookahead")
    assert ei.value.code == _ffi.PI_ERR_INVALID
    # unknown controller and wrong shapes: ValueError before any device call
    with pytest.raises(ValueError):
        eng.rollout(x0, 5, controller="greedy")
    with pytest.raises(ValueError):
        eng.lookahead(np.zeros((3, D + 1), F32))
    # a handle without values
    v, policy = eng.download()
    h = PolicyRollout(policy, eng.action_space, eng.bounds_low, eng.bounds_high, eng.grid_shape, eng._dynamics_cuda_src())
    for call in (lambda: h.lookahead(x0, 0.9), lambda: h.lookahead(np.zeros((0, D), F32), 0.9),
                 lambda: h.run(x0, 5, 0.9, controller="lookahead")):
        with pytest.raises(_ffi.EngineError) as ei:
            call()
        assert ei.value.code == _ffi.PI_ERR_INVALID and "pi_rollout_set_values" in str(ei.value)
    with pytest.raises(ValueError):
        h.set_values(v[:-1])
    with pytest.raises(ValueError):
        h.run(x0, 5, 0.9, controller="Lookahead")
    # still usable, and the ABI's null checks
    h.set_values(v)
    np.testing.assert_array_equal(h.lookahead(x0, F32(eng.config.gamma))[0], eng.lookahead(x0)[0])
    lib = _ffi.lib()
    assert lib.pi_rollout_lookahead(None, _ffi.ptr(x0), 1, 0.9, None, None) == _ffi.PI_ERR_INVALID
    assert lib.pi_rollout_lookahead(h._h, None, 1, 0.9, None, None) == _ffi.PI_ERR_INVALID
    assert lib.pi_rollout_lookahead(h._h, _ffi.ptr(x0), -1, 0.9, None, None) == _ffi.PI_ERR_INVALID
    assert lib.pi_rollout_lookahead(h._h, _ffi.ptr(x0), len(x0), 0.9, None, None) == _ffi.PI_OK
    assert lib.pi_rollout_set_values(h._h, None) == _ffi.PI_ERR_INVALID
    h.close()
    eng.close()


# ── 7. runner ──────────────────────────────────────────────────────────────────────────────────────────────────────

def test_runner_lookahead_rollout_summary_equals_pi_rollout(tmp_path, capsys):
    path = tmp_path / "cartpole_cuda_policy.npz"
    assert runners.main(["cartpole_cuda", "--bins", "8", "--save-path", str(path), "--no-plot", "--rollout",
                         "--rollout-controller", "lookahead", "--episodes", "16", "--steps", "50"]) == 0
    out = capsys.readouterr().out
    line = [ln for ln in out.splitlines() if ln.startswith("[=] rollout")]
    assert len(line) == 1 and "lookahead" in line[0]
    spec = envs.REGISTRY["cartpole"]
    pi = spec.cls.load(path)
    res = pi.rollout(runners.start_states(pi, 16, 42), 50, gamma=float(F32(spec.config().gamma)), controller="lookahead")
    expect = runners.format_rollout({"episodes": 16, "steps": 50, "mean_return": float(res.total_reward.mean()),
                                     "mean_discounted_return": float(res.discounted_return.mean()),
                                     "mean_length": float(res.length.mean()), "terminated": float(res.terminated.mean()),
                                     "controller": "lookahead"})
    assert line[0] == expect
