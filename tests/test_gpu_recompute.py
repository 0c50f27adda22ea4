"""Recompute mode (N7, include/dpb200.h: pi_create, DPB200_TABLE) against full-table mode, bit for bit.

In recompute mode the engine keeps no all-action table: the improvement pass recomputes every (state, action) row from
the plugin's dynamics, and the rows of a policy, expand_rows and the sharded exchange plan are rebuilt where the table
was read.  Full-table mode is the oracle here: the rest of the suite pins it to the reference's kernels.  Compared:
policy, V bits, PI iterations, sweeps and every improvement's change count, over real plugins (sinf / cosf / fmodf)
and the odd-D fixture; the improvement rule on adversarial values and on rewards that are NaN, -inf, -1e30, -0.0 and
exact duplicates; every row-producing path; and a grid whose all-action table is larger than the device."""
import importlib.util
import os
import shutil
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from dynamicprogramming_b200 import _ffi, envs
from dynamicprogramming_b200.engine import CudaPIConfig, _CudaPolicyIterationBase

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
_spec = importlib.util.spec_from_file_location("odd_dims", ROOT / "tests" / "fixtures" / "odd_dims.py")
odd = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(odd)

F32 = np.float32
U = 2.0 ** -24
DIMS = [1, 2, 3, 4, 5, 6]
MODES = ("full", "recompute")
# bins of the small grid each registry environment is solved on
ENV_BINS = {"pendulum": 41, "mountain_car": 41, "continuous_mountain_car": 41, "cartpole": 9, "cartpole_swingup": 9,
            "double_pendulum_swingup": 9, "overhead_crane": 9, "double_cartpole": 5, "double_cartpole_swingup": 5}


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def _mode(monkeypatch, mode):
    monkeypatch.setenv("DPB200_TABLE", mode)


def _solve(eng):
    """run()'s loop with every iteration's sweeps and change count recorded."""
    trace = []
    for _ in range(eng.config.max_pi_iter):
        eng.policy_evaluation()
        stable = eng.policy_improvement()
        trace.append((eng.last_eval_sweeps, eng.last_changed))
        if stable:
            break
    v, p = eng.download()
    return trace, p, bits(v).copy()


def _assert_same(got, want, what):
    assert got[0] == want[0], f"{what}: (sweeps, changed) per PI iteration"
    np.testing.assert_array_equal(got[1], want[1], err_msg=f"{what}: policy")
    np.testing.assert_array_equal(got[2], want[2], err_msg=f"{what}: value function bits")


def _stats_mode(eng):
    st = eng.engine_stats()
    return st["table_mode"], st["table_bytes"]


# ── 1. full runs ───────────────────────────────────────────────────────────────────────────────────────────────────

@pytest.mark.parametrize("name", sorted(envs.REGISTRY))
def test_run_in_recompute_mode_equals_full_mode_for_every_environment(name, monkeypatch):
    assert set(ENV_BINS) == set(envs.REGISTRY)
    spec = envs.REGISTRY[name]
    out = {}
    for mode in MODES:
        _mode(monkeypatch, mode)
        cfg = spec.config()
        cfg.max_eval_iter, cfg.max_pi_iter = 400, 6
        eng = envs.make(name, bins=ENV_BINS[name], config=cfg)
        eng.build_table()
        tm, tb = _stats_mode(eng)
        assert tm == mode and (tb == 0) == (mode == "recompute"), (tm, tb)
        out[mode] = _solve(eng)
        eng.close()
    _assert_same(out["recompute"], out["full"], name)


@pytest.mark.parametrize("D", DIMS)
def test_run_in_recompute_mode_equals_full_mode_for_the_odd_dims_fixture(D, monkeypatch):
    out = {}
    for mode in MODES:
        _mode(monkeypatch, mode)
        eng = odd.make(D)
        out[mode] = _solve(eng)
        eng.close()
    assert out["full"][0][-1][1] == 0, "the fixture converges"
    _assert_same(out["recompute"], out["full"], f"D={D}")


# ── 2. the improvement rule ────────────────────────────────────────────────────────────────────────────────────────

def _adversarial_values(N, seed):
    rng = np.random.default_rng(seed)
    V = (rng.choice([-1.0, 1.0], N) * 10.0 ** rng.uniform(-12, 12, N)).astype(F32)
    V[rng.random(N) < 0.05] = F32(0.0)
    V[rng.random(N) < 0.05] = F32(-0.0)
    return V


def _improve_once(eng, V, P0):
    eng.upload_values(V)
    eng.upload_policy(P0)
    stable = eng.policy_improvement()
    changed = eng.last_changed
    _, P1 = eng.download()
    eng.sweeps(1)                  # reads the rows the improvement wrote
    V1, _ = eng.download()
    return stable, changed, P1, bits(V1).copy()


@pytest.mark.parametrize("D", DIMS)
def test_one_improvement_from_adversarial_values_equals_full_mode(D, monkeypatch):
    out = {}
    for mode in MODES:
        _mode(monkeypatch, mode)
        eng = odd.make(D)
        N = eng.n_states
        P0 = np.random.default_rng(40 + D).integers(0, eng.n_actions, N).astype(np.int32)
        out[mode] = _improve_once(eng, _adversarial_values(N, 300 + D), P0)
        eng.close()
    assert out["recompute"][:2] == out["full"][:2]
    np.testing.assert_array_equal(out["recompute"][2], out["full"][2])
    np.testing.assert_array_equal(out["recompute"][3], out["full"][3])


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


def test_nan_inf_signed_zero_and_tied_rewards_pick_the_same_winner(monkeypatch):
    space = {"x": np.arange(16, dtype=F32), "y": np.linspace(-1, 1, 9, dtype=F32)}
    acts = np.arange(8, dtype=F32)
    out = {}
    for mode in MODES:
        _mode(monkeypatch, mode)
        rng = np.random.default_rng(5)
        eng = EdgeRewards(space, acts, CudaPIConfig(gamma=0.5))
        N = eng.n_states
        res = []
        for V in (np.zeros(N, F32), np.full(N, -1.4e-45, F32),
                  rng.choice(np.array([0.0, -0.0, -1.4e-45, 1.4e-45, 1e-40, -1e-40, 5.0, -5.0], F32), N)):
            res.append(_improve_once(eng, V.astype(F32), rng.integers(0, 8, N).astype(np.int32)))
        out[mode] = res
        eng.close()
    cls = (np.arange(16)[:, None] & 3).repeat(9, axis=1).ravel()
    for full, rc in zip(out["full"], out["recompute"]):
        assert rc[:2] == full[:2]
        np.testing.assert_array_equal(rc[2], full[2])
        np.testing.assert_array_equal(rc[3], full[3])
        assert (full[2][cls == 0] == 6).all() and (full[2][cls == 1] == 0).all() and (full[2][cls == 3] == 5).all()


# ── 3. every row-producing path ────────────────────────────────────────────────────────────────────────────────────

def _edited_odd(D):
    base = odd.plugin_class(D)

    class Edited(base):
        def _dynamics_cuda_src(self) -> str:
            src = super()._dynamics_cuda_src()
            assert odd.ACTION_COST in src
            return src.replace(odd.ACTION_COST, "0.2f")

    return Edited


def _row_paths(D, monkeypatch, mode):
    """Everything that produces rows, in one engine per storage order: expand_rows, upload_policy (+ sweeps),
    upload_policy_local (pipelined with the plane-staged sweep at D >= 4), warm_start, retrain with the same and an
    edited text, run()."""
    _mode(monkeypatch, mode)
    res = {}
    rng = np.random.default_rng(11 + D)
    layouts = ["ref", "0"] + (["0,1"] if D >= 4 else [])
    for fast in layouts:
        monkeypatch.setenv("DPB200_FAST_DIM", fast)
        if fast == "0,1":
            monkeypatch.setenv("DPB200_PLANE", "force:0,0,2,2,2")
        eng = odd.make(D)
        eng.build_table()
        N, A = eng.n_states, eng.n_actions
        r = res.setdefault(fast, [])
        for a in range(A):
            r.append(tuple(np.ascontiguousarray(x).view(np.uint8).copy() for x in eng.expand_rows(a)))
        r.append(tuple(np.ascontiguousarray(x).view(np.uint8).copy() for x in eng.expand_rows(A - 1, N // 3, N // 2)))
        P = rng.integers(0, A, N).astype(np.int32)
        eng.upload_policy(P)
        eng.sweeps(3)
        r.append(bits(eng.download()[0]).copy())
        if fast == "0,1":
            assert "ps_sweep" in eng.eval_kernel_info()["kernel"]
        eng.upload_policy_local(eng.to_internal_order(rng.integers(0, A, N).astype(np.int32)))
        eng.sweeps(3)
        r.append(bits(eng.download()[0]).copy())
        coarse = tuple(max(2, s // 2) for s in odd.SHAPES[D])
        src = rng.standard_normal(int(np.prod(coarse))).astype(F32)
        ws = eng.warm_start((src, eng.bounds_low, eng.bounds_high, np.array(coarse)))
        r.append(ws["changed"])
        eng.sweeps(2)
        r.append(tuple(bits(x).copy() if x.dtype == F32 else x.copy() for x in eng.download()))
        assert eng.retrain() is False
        r.append(_solve(eng))
        eng.__class__ = _edited_odd(D)
        assert eng.retrain() is True
        r.append(_solve(eng))
        assert _stats_mode(eng)[0] == mode
        eng.close()
        monkeypatch.delenv("DPB200_PLANE", raising=False)
    return res


def _flatten(x):
    if isinstance(x, (list, tuple)):
        for y in x:
            yield from _flatten(y)
    else:
        yield x


@pytest.mark.parametrize("D", DIMS)
def test_every_row_producing_path_equals_full_mode(D, monkeypatch):
    want = _row_paths(D, monkeypatch, "full")
    got = _row_paths(D, monkeypatch, "recompute")
    assert want.keys() == got.keys()
    for fast in want:
        w, g = list(_flatten(want[fast])), list(_flatten(got[fast]))
        assert len(w) == len(g)
        for i, (a, b) in enumerate(zip(w, g)):
            if isinstance(a, np.ndarray):
                np.testing.assert_array_equal(b, a, err_msg=f"D={D} DPB200_FAST_DIM={fast} item {i}")
            else:
                assert a == b, (D, fast, i)


# ── 4. a grid whose all-action table does not fit on the device ────────────────────────────────────────────────────

BIG_SHAPE = (20, 20, 20, 20, 20, 16)      # 25.6 M states
BIG_ACTIONS = np.linspace(-1.0, 1.0, 256, dtype=F32)


def _big(monkeypatch, mode, max_eval_iter=20):
    _mode(monkeypatch, mode)
    monkeypatch.delenv("DPB200_FAST_DIM", raising=False)
    space = {f"x{k}": np.linspace(*odd.RANGES[k], n, dtype=F32) for k, n in enumerate(BIG_SHAPE)}
    cfg = CudaPIConfig(gamma=odd.GAMMA, theta=1e-5, max_eval_iter=max_eval_iter, max_pi_iter=1)
    return odd.plugin_class(6)(space, BIG_ACTIONS, cfg)


def _host_rows(eng, a, ref_states):
    """host_rows of tests/test_gpu_odd_dims.py for the states `ref_states` only and the action value of index a."""
    D = eng.N_DIMS
    C = 1 << D
    shape = [int(s) for s in eng.grid_shape]
    stride = np.array(eng.strides, np.int64)
    coords = np.stack(np.unravel_index(ref_states, shape), axis=1)
    states = np.stack([eng._axes[d][coords[:, d]] for d in range(D)], axis=1).astype(F32)
    nx, r, term = odd.step_numpy(states, eng.action_space[a])
    absorbing = odd.terminal_mask(states)
    code = np.where(absorbing, 2, np.where(term, 1, 0)).astype(np.uint8)
    live = code == 0
    n = len(ref_states)
    idx = np.where(code == 1, -1, -2).astype(np.int64)[:, None].repeat(C, axis=1)
    w = np.zeros((n, C), F32)
    base = np.zeros(int(live.sum()), np.int64)
    fr = np.empty((int(live.sum()), D), F32)
    for d in range(D):
        lo, hi = F32(eng.bounds_low[d]), F32(eng.bounds_high[d])
        pn = ((nx[live, d] - lo).astype(F32) / F32(hi - lo)).astype(F32)
        pn = (pn * F32(shape[d] - 1)).astype(F32)
        pn = np.maximum(F32(0), np.minimum(pn, F32(shape[d] - 1)))
        i = np.minimum(pn.astype(np.int64), shape[d] - 2)
        base += i * stride[d]
        fr[:, d] = (pn - i.astype(F32)).astype(F32)
    for c in range(C):
        idx[live, c] = base + sum(((c >> d) & 1) * int(stride[d]) for d in range(D))
        wc = np.ones(len(base), F32)
        for d in range(D):
            wc = (wc * (fr[:, d] if (c >> d) & 1 else (F32(1) - fr[:, d]).astype(F32))).astype(F32)
        w[live, c] = wc
    return idx, w, np.where(absorbing, F32(0), r).astype(F32), code


def test_a_table_larger_than_the_device_solves_in_recompute_mode(monkeypatch):
    import torch

    total = torch.cuda.get_device_properties(0).total_memory
    N = int(np.prod(BIG_SHAPE))
    assert len(BIG_ACTIONS) * 8 * 4 * N > total, "the all-action table must not fit"
    eng = _big(monkeypatch, "auto")
    eng.build_table()
    tm, tb = _stats_mode(eng)
    assert (tm, tb) == ("recompute", 0)
    eng.policy_evaluation()
    V, P0 = eng.download()
    eng.policy_improvement()
    _, P1 = eng.download()
    rng = np.random.default_rng(3)
    s0 = int(rng.integers(0, N - 256))
    sample = np.arange(s0, s0 + 256)
    for a in (0, 97, 255):
        got = eng.expand_rows(a, s0, 256)
        want = _host_rows(eng, a, sample)
        for x, y in zip(got, want):
            np.testing.assert_array_equal(np.ascontiguousarray(x).view(np.uint8),
                                          np.ascontiguousarray(y.astype(x.dtype)).view(np.uint8))
    # the improved policy on the sampled states against float64 Q-values of every action
    rows = [_host_rows(eng, a, sample) for a in range(len(BIG_ACTIONS))]
    idx, w, r, code = (np.stack([rw[k] for rw in rows]) for k in range(4))
    Vd = V.astype(np.float64)
    wv = w.astype(np.float64) * Vd[np.maximum(idx, 0)]
    wv[code != 0] = 0.0
    g = float(F32(odd.GAMMA))
    q = r.astype(np.float64) + g * wv.sum(axis=2)
    tol = ((1 << 6) + 2) * U * (g * np.abs(wv).sum(axis=2) + np.abs(r.astype(np.float64)))
    j = np.arange(len(sample))
    p1 = P1[sample]
    best = q.argmax(axis=0)
    live = code[0] != 2
    gap = q[best, j] - q[p1, j]
    assert (gap[live] <= (tol[best, j] + tol[p1, j])[live]).all(), float(gap[live].max())
    np.testing.assert_array_equal(p1[~live], P0[sample][~live])
    eng.close()
    with pytest.raises(_ffi.EngineError) as err:
        _big(monkeypatch, "full")
    assert err.value.code == _ffi.PI_ERR_CUDA


def test_a_bad_table_mode_is_invalid(monkeypatch):
    _mode(monkeypatch, "sometimes")
    with pytest.raises(_ffi.EngineError) as err:
        odd.make(2)
    assert err.value.code == _ffi.PI_ERR_INVALID and "DPB200_TABLE" in str(err.value)


# ── 5. sharded ─────────────────────────────────────────────────────────────────────────────────────────────────────

def test_sharded_run_in_recompute_mode_is_bit_identical_on_two_gpus():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", DPB200_TABLE="recompute")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29613", str(ROOT / "scripts" / "multi_gpu_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "FAIL" not in res.stdout


# ── 6. compute-sanitizer ───────────────────────────────────────────────────────────────────────────────────────────

SAN = shutil.which("compute-sanitizer") or str(Path(shutil.which("nvcc") or "nvcc").resolve().parent / "compute-sanitizer")


def _sanitizer_usable() -> bool:
    if not Path(SAN).exists():
        return False
    try:
        res = subprocess.run([SAN, "--version"], capture_output=True, text=True, timeout=60)
    except (OSError, subprocess.TimeoutExpired):
        return False
    return res.returncode == 0 and "Compute Sanitizer" in res.stdout


@pytest.mark.parametrize("tool", ["memcheck", "racecheck"])
def test_recompute_kernels_are_clean_under_compute_sanitizer(tool):
    """pi_improve_recompute and pi_policy_rows (shared-memory counters: racecheck too) through build, improvement,
    policy upload and sweeps (scripts/sanitize_target.py recompute)."""
    if not _sanitizer_usable():
        pytest.skip("compute-sanitizer is not installed or cannot run here")
    cmd = [SAN, "--tool", tool, "--error-exitcode", "1", sys.executable, str(ROOT / "scripts" / "sanitize_target.py"),
           "recompute"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, DPB200_CACHE="off"))
    tail = (res.stdout + res.stderr)[-3000:]
    assert res.returncode == 0, tail
    assert "SANITIZE_TARGET_OK" in res.stdout, tail
    assert ("ERROR SUMMARY: 0 errors" in tail) or ("RACECHECK SUMMARY: 0 hazards" in tail), tail
