"""Warm start from another grid's value function (include/dpb200.h: pi_prolong_values; engine.warm_start).

* The prolongation equals a numpy restatement bit for bit: lookup_numpy of tests/test_gpu_odd_dims.py with V[flat] in
  place of actions[policy[flat]], evaluated at states_space, on every fixture dimensionality and on the overhead crane
  at two bin counts; from coarser, finer, equal, differently bounded (clamped on both sides) sources and a source with a
  dimension of 2 nodes; in every storage order.  Both V buffers hold the same bits; absorbing states keep their values.
* warm_start(src) is pi_prolong_values + policy_improvement(): a twin engine that uploads the restated V and improves
  gets the same policy and the same run().
* A warm-started run() is a solution: within the bound of an exact solve of its own policy, greedy with respect to its
  V, and its policy's exact values agree with the cold run's within a bound derived from theta, gamma and rounding.
* Errors leave the engine usable; retrain() after a warm start equals a fresh engine; the runner's flags; the
  sanitizer family; a sharded warm start on two GPUs."""
import ctypes as C
import importlib.util
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from dynamicprogramming_b200 import _ffi, envs, runners
from dynamicprogramming_b200.engine import CudaPIConfig

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]

_spec = importlib.util.spec_from_file_location("odd_dims", ROOT / "tests" / "fixtures" / "odd_dims.py")
odd = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(odd)
_spec2 = importlib.util.spec_from_file_location("odd_dims_tests", ROOT / "tests" / "test_gpu_odd_dims.py")
odt = importlib.util.module_from_spec(_spec2)
_spec2.loader.exec_module(odt)

F32 = np.float32
DIMS = [1, 2, 3, 4, 5, 6]
ENGINE_ENV = ("DPB200_FAST_DIM", "DPB200_PLANE", "DPB200_XLINE", "DPB200_PAIR", "DPB200_PERSIST")


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def interp_numpy(values, lo, hi, shape, pts):
    """lookup_numpy with V[flat] in place of actions[policy[flat]]: an identity policy over the values as actions."""
    values = np.asarray(values, F32)
    return odt.lookup_numpy(np.arange(values.size), values, lo, hi, shape, pts)


def _env(monkeypatch, **env):
    for k in ENGINE_ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def _prolong(eng, values, lo, hi, shape):
    grid = _ffi.PiGrid()
    grid.n_dims = len(shape)
    for d in range(len(shape)):
        grid.shape[d], grid.lo[d], grid.hi[d] = int(shape[d]), float(lo[d]), float(hi[d])
    v = np.ascontiguousarray(values, F32)
    ms = C.c_float()
    _ffi.check(_ffi.lib().pi_prolong_values(eng._engine, C.byref(grid), _ffi.ptr(v), C.byref(ms)))
    return ms.value


def _sources(eng, seed):
    """(name, values, lo, hi, shape): coarser, finer, equal, shifted / narrowed bounds (nodes outside on both sides),
    and a coarser grid with a dimension of 2 nodes."""
    rng = np.random.default_rng(seed)
    D = eng.N_DIMS
    lo, hi = eng.bounds_low.astype(F32), eng.bounds_high.astype(F32)
    shape = np.array(eng.grid_shape, np.int64)
    span = (hi - lo).astype(F32)
    out = []
    for name, shp, l, h in (
            ("coarser", np.maximum(2, (shape + 1) // 2), lo, hi),
            ("finer", shape * 2 - 1, lo, hi),
            ("equal", shape, lo, hi),
            ("bounds", np.maximum(2, shape - 1), (lo + F32(0.3) * span).astype(F32), (hi - F32(0.2) * span).astype(F32)),
            ("two_nodes", np.where(np.arange(D) == D - 1, 2, np.maximum(2, shape // 2 + 1)), lo, hi)):
        n = int(np.prod(shp))
        out.append((name, (rng.standard_normal(n) * 10).astype(F32), l, h, shp))
    return out


def _check_prolongation(eng, sources, absorbing):
    """Each source prolonged once; both buffers; absorbing states keep what they held (on the first source the values
    the engine was given at construction; afterwards random values uploaded into the current buffer)."""
    rng = np.random.default_rng(11)
    for k, (name, vals, lo, hi, shp) in enumerate(sources):
        before, _ = eng.download()
        ms = _prolong(eng, vals, lo, hi, shp)
        assert ms >= 0
        got, _ = eng.download()
        want = interp_numpy(vals, lo, hi, shp, eng.states_space)
        live = ~absorbing
        np.testing.assert_array_equal(bits(got[live]), bits(want[live]), err_msg=name)
        np.testing.assert_array_equal(bits(got[absorbing]), bits(before[absorbing]), err_msg=name)
        v0, v1 = eng.d_value_function.get(), eng.d_new_value_function.get()
        np.testing.assert_array_equal(bits(v0), bits(got))
        if k == 0:   # both buffers held the same values before: they do after, everywhere
            np.testing.assert_array_equal(bits(v1), bits(v0), err_msg=name)
        else:
            np.testing.assert_array_equal(bits(v1[live]), bits(v0[live]), err_msg=name)
        eng.upload_values(rng.standard_normal(eng.n_states).astype(F32))


@pytest.mark.parametrize("D", DIMS)
def test_prolongation_is_bit_exact_in_every_storage_order(D, monkeypatch):
    for order in ["ref", "0", "auto"] + (["0,1"] if D >= 4 else []):
        _env(monkeypatch, DPB200_FAST_DIM=order)
        eng = odd.make(D)
        eng.build_table()
        if order != "auto" and order != "ref":
            assert eng.layout()["fast_dim"] == 0
        absorbing = odd.terminal_mask(eng.states_space)
        assert absorbing.any()
        v, _ = eng.download()
        np.testing.assert_array_equal(v[absorbing], F32(odd.TERMINAL_VALUE))
        _check_prolongation(eng, _sources(eng, 40 + D), absorbing)
        eng.close()


@pytest.mark.parametrize("bins", [11, 15])
def test_prolongation_on_the_crane_keeps_goal_values(bins, monkeypatch):
    """The crane's goal states are in its terminal mask and hold 1/(1 - gamma) from set_values: they keep it."""
    for order in ["ref", "auto"]:
        _env(monkeypatch, DPB200_FAST_DIM=order)
        eng = envs.make("overhead_crane", bins=bins)
        eng.build_table()
        absorbing = eng._terminal_mask_host.astype(bool)
        goal = eng._goal_mask
        assert goal.any() and (absorbing & ~goal).any()
        v, _ = eng.download()
        np.testing.assert_array_equal(v[goal], F32(1.0 / (1.0 - eng.config.gamma)))
        _check_prolongation(eng, _sources(eng, bins), absorbing)
        eng.close()


def _coarse_solution(D, cfg=None):
    """The fixture's plugin solved on a coarser grid of the same box (dimensions of 2 nodes stay 2)."""
    shape = [max(2, (n + 1) // 2) for n in odd.SHAPES[D]]
    bins = {f"x{k}": np.linspace(odd.RANGES[k][0], odd.RANGES[k][1], n, dtype=F32) for k, n in enumerate(shape)}
    eng = odd.plugin_class(D)(bins, odd.ACTIONS, cfg or CudaPIConfig(gamma=odd.GAMMA, theta=1e-5, max_eval_iter=10_000,
                                                                      max_pi_iter=50))
    eng.run()
    assert eng.converged
    return eng


def _restated(eng, src):
    """The V a warm start gives `eng` (a fresh engine): the restatement on live states, the held values on absorbing."""
    v, _ = eng.download()
    absorbing = odd.terminal_mask(eng.states_space)
    want = interp_numpy(src.value_function, src.bounds_low, src.bounds_high, src.grid_shape, eng.states_space)
    return np.where(absorbing, v, want).astype(F32)


@pytest.mark.parametrize("D,env", [(2, {}), (4, {}), (6, {}), (3, {}),
                                   (4, {"DPB200_FAST_DIM": "0,1", "DPB200_PLANE": "force:0,0,2,2,2"}),
                                   (6, {"DPB200_FAST_DIM": "0,1", "DPB200_PLANE": "force:0,0,2,2,2"})])
def test_warm_start_is_prolongation_then_improvement(D, env, monkeypatch):
    _env(monkeypatch)
    src = _coarse_solution(D)
    _env(monkeypatch, **env)
    a = odd.make(D)
    b = odd.make(D)
    if env:
        a.build_table()
        assert "ps_sweep" in a.eval_kernel_info()["kernel"]
    ws = a.warm_start(src)
    b.build_table()
    b.upload_values(_restated(b, src))
    b.policy_improvement()
    assert ws["changed"] == b.last_changed > 0 and ws["prolong_ms"] >= 0
    va, pa = a.download()
    vb, pb = b.download()
    np.testing.assert_array_equal(pa, pb)
    np.testing.assert_array_equal(bits(va), bits(vb))
    a.run()
    b.run()
    assert (a.pi_iterations, a.total_eval_sweeps) == (b.pi_iterations, b.total_eval_sweeps)
    np.testing.assert_array_equal(a.policy, b.policy)
    np.testing.assert_array_equal(bits(a.value_function), bits(b.value_function))


def _exact_values(rows, P, N, g):
    idx, w, r, code = (x[P, np.arange(N)] for x in rows)
    live = code == 0
    C_ = idx.shape[1]
    rr = np.repeat(np.arange(N)[live], C_)
    A = sp.identity(N, format="csr") - sp.csr_matrix((g * w[live].astype(np.float64).ravel(), (rr, idx[live].ravel())),
                                                     shape=(N, N))
    b = np.where(code == 2, odd.TERMINAL_VALUE, r.astype(np.float64))
    return spla.spsolve(A.tocsc(), b)


@pytest.mark.parametrize("D", DIMS)
def test_warm_run_is_a_solution_and_agrees_with_the_cold_run(D, monkeypatch):
    """For each run (warm, cold) let eps be the fma-chain bound of its backups (q_values) and
    b = (gamma theta + eps) / (1 - gamma) the bound |V - V_pi| of test_run_matches_an_exact_solve_of_its_policy.
    The policy is greedy with respect to V up to delta = max_s (tol[best] + tol[P]) (asserted below).  Then
    V* - V_pi = (T*V* - T*V) + (T*V - T_pi V) + (T_pi V - T_pi V_pi) <= gamma |V* - V| + delta + gamma |V - V_pi|
    and |V* - V| <= |V* - V_pi| + b give 0 <= V* - V_pi <= (delta + 2 gamma b) / (1 - gamma) =: B.  Both exact value
    functions lie in [V* - B, V*], so |V_pi_warm - V_pi_cold| <= max(B_warm, B_cold)."""
    _env(monkeypatch, DPB200_PLANE="off", DPB200_XLINE="off", DPB200_PAIR="off", DPB200_PERSIST="off")
    cfg = CudaPIConfig(gamma=odd.GAMMA, theta=1e-5, max_eval_iter=10_000, max_pi_iter=50)
    src = _coarse_solution(D, cfg)
    warm = odd.make(D, cfg)
    warm.build_table()
    rows = odt.all_host_rows(warm)
    warm.warm_start(src)
    warm.run()
    assert warm.converged
    cold = odd.make(D, cfg)
    cold.run()
    assert cold.converged
    N = warm.n_states
    s = np.arange(N)
    g = float(F32(cfg.gamma))
    theta = float(F32(cfg.theta)) * (1 + 2.0 ** -22)
    bounds, exact = [], []
    for run in (warm, cold):
        V, P = run.value_function, run.policy
        v_pi = _exact_values(rows, P, N, g)
        q, tol = odt.q_values(rows, V, cfg.gamma)
        eps = 1.01 * tol[P, s].max()
        b = (g * theta + eps) / (1 - g)
        assert np.abs(V.astype(np.float64) - v_pi).max() <= b
        best = q.argmax(axis=0)
        gap = q[best, s] - q[P, s]
        assert (gap <= tol[best, s] + tol[P, s]).all(), float(gap.max())
        delta = float((tol[best, s] + tol[P, s]).max())
        bounds.append((delta + 2 * g * b) / (1 - g))
        exact.append(v_pi)
        np.testing.assert_array_equal(V[odd.terminal_mask(run.states_space)], F32(odd.TERMINAL_VALUE))
    assert np.abs(exact[0] - exact[1]).max() <= max(bounds), (float(np.abs(exact[0] - exact[1]).max()), bounds)


def test_errors_leave_the_engine_usable(monkeypatch):
    _env(monkeypatch)
    D = 3
    want = odd.make(D)
    want.run()
    eng = odd.make(D)
    shape = np.array(odd.SHAPES[D])
    lo, hi = eng.bounds_low, eng.bounds_high
    vals = np.zeros(int(np.prod(shape)), F32)
    with pytest.raises(_ffi.EngineError, match="pi_build_table"):
        _prolong(eng, vals, lo, hi, shape)                           # before the table exists
    eng.build_table()
    with pytest.raises(_ffi.EngineError, match="dimensions"):
        eng.warm_start((np.zeros(int(np.prod(shape[:2])), F32), lo[:2], hi[:2], shape[:2]))
    bad = shape.copy()
    bad[1] = 1
    with pytest.raises(_ffi.EngineError, match=">= 2 nodes"):
        eng.warm_start((np.zeros(int(np.prod(bad)), F32), lo, hi, bad))
    lo2 = lo.copy()
    lo2[2] = hi[2]
    with pytest.raises(_ffi.EngineError, match="lo\\[2\\] >= hi\\[2\\]"):
        eng.warm_start((vals, lo2, hi, shape))
    with pytest.raises(_ffi.EngineError, match="values for a grid"):
        eng.warm_start((vals[:-1], lo, hi, shape))
    eng.run()
    assert (eng.pi_iterations, eng.total_eval_sweeps) == (want.pi_iterations, want.total_eval_sweeps)
    np.testing.assert_array_equal(eng.policy, want.policy)
    np.testing.assert_array_equal(bits(eng.value_function), bits(want.value_function))


def test_retrain_after_a_warm_start_equals_a_fresh_engine(monkeypatch):
    _env(monkeypatch)
    D = 4
    src = _coarse_solution(D)
    eng = odd.make(D)
    eng.warm_start(src)
    eng.sweeps(5)
    eng.retrain()
    eng.run()
    fresh = odd.make(D)
    fresh.run()
    assert (eng.pi_iterations, eng.total_eval_sweeps) == (fresh.pi_iterations, fresh.total_eval_sweeps)
    np.testing.assert_array_equal(eng.policy, fresh.policy)
    np.testing.assert_array_equal(bits(eng.value_function), bits(fresh.value_function))


def test_warm_start_accepts_a_path_an_instance_and_a_tuple(monkeypatch, tmp_path):
    _env(monkeypatch)
    D = 2
    src = _coarse_solution(D)
    src.save(tmp_path / "coarse")
    loaded = odd.plugin_class(D).load(tmp_path / "coarse.npz")
    out = []
    for source in (src, tmp_path / "coarse.npz", loaded,
                   (src.value_function, src.bounds_low, src.bounds_high, src.grid_shape)):
        eng = odd.make(D)
        eng.warm_start(source)
        out.append(eng.download())
        eng.close()
    for v, p in out[1:]:
        np.testing.assert_array_equal(bits(v), bits(out[0][0]))
        np.testing.assert_array_equal(p, out[0][1])


def test_runner_warm_start_flags(tmp_path, capsys):
    plain = tmp_path / "plain.npz"
    assert runners.main(["cartpole_cuda", "--bins", "8", "--save-path", str(plain), "--episodes", "2"]) == 0
    out = capsys.readouterr().out
    assert "[=] solve at" not in out and "Training new policy" in out and out.count("-> action") == 2
    warm = tmp_path / "warm.npz"
    assert runners.main(["cartpole_cuda", "--bins", "8", "--warm-start-bins", "5", "--save-path", str(warm),
                         "--episodes", "2"]) == 0
    out = capsys.readouterr().out
    lines = [ln for ln in out.splitlines() if ln.startswith("[=] solve at")]
    assert len(lines) == 2 and lines[0].startswith("[=] solve at 5 bins |") and lines[1].startswith("[=] solve at 8 bins |")
    assert "evaluation sweeps" in lines[1] and lines[1].endswith(" s")
    assert np.load(warm)["states_space"].shape == (8 ** 4, 4)
    again = tmp_path / "again.npz"
    assert runners.main(["cartpole_cuda", "--bins", "9", "--warm-start-from", str(warm), "--save-path", str(again),
                         "--episodes", "0"]) == 0
    out = capsys.readouterr().out
    lines = [ln for ln in out.splitlines() if ln.startswith("[=] solve at")]
    assert len(lines) == 1 and lines[0].startswith("[=] solve at 9 bins |")
    assert np.load(again)["policy"].shape == (9 ** 4,)


def test_warm_start_family_under_memcheck():
    spec = importlib.util.spec_from_file_location("sanitizer_tests", ROOT / "tests" / "test_gpu_sanitizer.py")
    san_tests = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(san_tests)
    if not san_tests._sanitizer_usable():
        pytest.skip("compute-sanitizer is not installed or cannot run here")
    san = san_tests.SAN
    cmd = [san, "--tool", "memcheck", "--error-exitcode", "1", sys.executable, str(ROOT / "scripts" / "sanitize_target.py"),
           "warm_start"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, DPB200_CACHE="off"))
    tail = (res.stdout + res.stderr)[-3000:]
    assert res.returncode == 0 and "SANITIZE_TARGET_OK" in res.stdout and "ERROR SUMMARY: 0 errors" in tail, tail


def test_sharded_warm_start_is_bit_identical_on_two_gpus():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29613", str(ROOT / "scripts" / "warm_start_multi_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "FAIL" not in res.stdout and "OK" in res.stdout
