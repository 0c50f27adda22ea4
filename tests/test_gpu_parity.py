"""Parity tests proper: the CUDA engine (through the C ABI) against what the
reference's own kernels compute (tests/golden/reference_parity.json) — bit-exact for
transition indices, weights, rewards, value functions, policies, sweep counts —
and against the reference's golden files and the CPU oracle at tolerance."""
import numpy as np
import pytest

from dynamicprogramming_b200 import envs

pytestmark = pytest.mark.gpu

SMALL = {"pendulum": 41, "mountain_car": 50, "continuous_mountain_car": 50, "cartpole": 9, "cartpole_swingup": 9,
         "double_pendulum_swingup": 9, "overhead_crane": 9, "double_cartpole": 5, "double_cartpole_swingup": 6}


@pytest.mark.parametrize("env", sorted(SMALL))
def test_transition_rows_are_bit_exact(env, reference):
    """Indices, weights, reward and `terminated` of every (state, action) row
    equal what the reference's step_dynamics + get_barycentric_Nd produce."""
    eng = envs.make(env, bins=SMALL[env])
    term = eng._terminal_mask_host.astype(bool)
    live = ~term
    for a in range(eng.n_actions):
        idx, w, r, t = eng.expand_rows(a)
        assert (t[term] == 2).all()                                  # absorbing rows are flagged
        reference.check(f"action {a} terminated", t[live] == 1)
        ok = live & (t != 1)
        reference.check(f"action {a} idx", idx[ok])
        reference.check(f"action {a} w", w[ok])
        reference.check(f"action {a} reward", r[live])
    eng.close()


@pytest.mark.parametrize("env", sorted(SMALL))
def test_single_sweep_and_improvement_are_bit_exact(env, reference):
    eng = envs.make(env, bins=SMALL[env])
    N, A = eng.n_states, eng.n_actions
    rng = np.random.default_rng(3)
    V0 = (rng.standard_normal(N) * 10).astype(np.float32)
    for a in list(range(min(A, 3))) + [A - 1]:
        pol = np.full(N, a, dtype=np.int32)
        eng.upload_policy(pol)
        eng.upload_values(V0)
        delta, _ = eng.sweeps(1)
        v_mine, _ = eng.download()
        reference.check(f"sweep under policy {a}", v_mine)
        assert np.float32(delta) == np.abs(v_mine - V0).max()         # fused residual == max|new_V - V|
    # mixed policy
    pol = rng.integers(0, A, N).astype(np.int32)
    eng.upload_policy(pol)
    eng.upload_values(V0)
    eng.sweeps(1)
    v_mine, _ = eng.download()
    reference.check("sweep under the mixed policy", v_mine)
    # improvement from the same V
    eng.upload_policy(np.zeros(N, dtype=np.int32))
    eng.upload_values(V0)
    stable = eng.policy_improvement()
    _, p_mine = eng.download()
    reference.check("improved policy", p_mine)
    assert stable == bool((p_mine == 0).all())
    assert eng.last_changed == int((p_mine != 0).sum())
    eng.close()


RUNS = [("mountain_car", 200, None), ("continuous_mountain_car", 200, None), ("pendulum", 200, None),
        ("cartpole", 20, None), ("cartpole_swingup", 10, 8), ("double_pendulum_swingup", 12, 6),
        ("overhead_crane", 12, 6), ("double_cartpole", 6, 6), ("double_cartpole_swingup", 8, 4)]


@pytest.mark.parametrize("env,bins,max_pi", RUNS)
def test_full_policy_iteration_is_bit_identical_to_the_reference(env, bins, max_pi, reference):
    """run(): same number of PI iterations and sweeps, identical policy, identical V bits."""
    spec = envs.REGISTRY[env]
    cfg = spec.config()
    if max_pi:
        cfg.max_pi_iter = max_pi
    eng = spec.make(bins=bins, config=cfg)
    eng.run()
    reference.check_run(eng)
    assert eng.value_function.dtype == np.float32 and eng.policy.dtype == np.int32
    assert not hasattr(eng, "d_value_function")                       # VRAM released like the reference


@pytest.mark.parametrize("env,min_agree,max_outliers", [("continuous_mountain_car", 0.999, 0), ("mountain_car", 0.995, 40)])
def test_converged_result_matches_the_reference_golden_files(golden_dir, env, min_agree, max_outliers):
    """The two artefacts the reference ships (trained on the author's GPU)."""
    g = np.load(golden_dir / f"{env}_golden.npz")
    eng = envs.make(env)
    eng.run()
    assert float(np.mean(eng.policy == g["policy"])) >= min_agree
    V = g["value_function"]
    rel = np.abs(eng.value_function - V) / np.maximum(np.abs(V), 1e-6)
    assert int((rel > 1e-5).sum()) <= max_outliers, float(rel.max())   # north_star: V within 1e-5 relative


@pytest.mark.parametrize("env,bins", [("pendulum", 64), ("cartpole", 11), ("double_cartpole_swingup", 5)])
def test_engine_agrees_with_the_cpu_oracle(env, bins):
    """Cross-check of the two oracles: CPU restatement vs CUDA engine (tolerance:
    libm vs CUDA transcendentals; V within 1e-5 relative on >= 99.5 % of states)."""
    from oracle import cpu_oracle

    spec = envs.REGISTRY[env]
    cfg = spec.config()
    cfg.max_pi_iter = 3
    eng = spec.make(bins=bins, config=cfg)
    eng.run()
    o = cpu_oracle.from_engine_env(env, bins=bins, config=cfg)
    o.run()
    rel = np.abs(eng.value_function - o.value_function) / np.maximum(np.abs(o.value_function), 1e-3)
    assert np.mean(rel < 1e-5) >= 0.995, float(np.mean(rel < 1e-5))
    assert np.mean(eng.policy == o.policy) >= 0.99
