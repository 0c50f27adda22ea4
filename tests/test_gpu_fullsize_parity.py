"""Bit-for-bit parity with what the reference's own kernels compute (tests/golden/reference_parity.json) AT BASELINE.json's sizes:
K2 (Continuous Mountain Car --bins 400, also with a 201-action grid) and K3 (CartPole --bins 30) complete run()s;
K4 (Double Pendulum swing-up --bins 50) and K5 (Double CartPole swing-up --bins 20, 64 M states) one improvement
pass and one evaluation sweep under the mixed policy of PI iteration 1 with the DEFAULT-selected sweep kernel
(and with every other sweep family forced), slab-wise transition rows of K5, and K5 --bins 12 (the autoresearch
trial workload, runners/trial_runner.sh:33-60) run to a stable policy.
Reference: src/cuda_policy_iteration.py:212-283, :616-691, :1044-1123, host loop :300-370."""
import numpy as np
import pytest

from dynamicprogramming_b200 import envs

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("env,bins,n_actions", [("continuous_mountain_car", 400, None), ("continuous_mountain_car", 400, 201),
                                                ("cartpole", 30, None)])
def test_complete_run_at_baseline_size_matches_the_reference(env, bins, n_actions, reference):
    spec = envs.REGISTRY[env]
    actions = None
    if n_actions is not None:
        actions = np.linspace(float(spec.actions.min()), float(spec.actions.max()), n_actions).astype(np.float32)
    eng = spec.make(bins=bins, actions=actions)
    eng.run()
    reference.check_run(eng)


def _mixed_policy(env, bins, sweeps=50):
    """Engine after `sweeps` sweeps of the initial policy and one improvement pass."""
    eng = envs.make(env, bins=bins)
    eng.build_table()
    eng.sweeps(sweeps)
    eng.policy_improvement()
    return eng


@pytest.mark.parametrize("env,bins,kernels", [("double_pendulum_swingup", 50, "default"), ("double_pendulum_swingup", 50, "gather"),
                                              ("double_pendulum_swingup", 50, "aot"), ("double_cartpole_swingup", 20, "default"),
                                              ("double_cartpole_swingup", 20, "gather"), ("double_cartpole_swingup", 20, "plane"),
                                              ("double_cartpole_swingup", 20, "plane_one"), ("double_cartpole_swingup", 20, "aot")])
def test_improvement_and_sweep_at_baseline_size_match_the_reference(env, bins, kernels, reference, monkeypatch):
    """K4 / K5: the improvement pass (policy bits) and one sweep under the resulting mixed policy (V bits), with the
    kernel the engine selects by default — the one bench.py times — and with each sweep family pinned."""
    if kernels == "gather":
        monkeypatch.setenv("DPB200_PLANE", "off")
        monkeypatch.setenv("DPB200_XLINE", "off")
    elif kernels == "plane":
        monkeypatch.setenv("DPB200_PLANE", "force")              # item mode (two states per thread)
    elif kernels == "plane_one":
        monkeypatch.setenv("DPB200_PLANE", "force:0,0,2,2,0")    # one state per thread
    elif kernels == "aot":
        monkeypatch.setenv("DPB200_PLANE", "off")
        monkeypatch.setenv("DPB200_XLINE", "off")
        monkeypatch.setenv("DPB200_PAIR", "off")
    eng = _mixed_policy(env, bins)
    info = eng.eval_kernel_info()
    if kernels == "default" and env == "double_cartpole_swingup":
        assert "ps_sweep" in info["kernel"] or "gp_sweep" in info["kernel"], info     # the JIT sweeps bench.py times
    if kernels in ("plane", "plane_one") and env == "double_cartpole_swingup":
        assert info["plane"] and ("pack 2" in info["kernel"]) == (kernels == "plane"), info
    if kernels == "aot":
        assert "eval_sweep_kernel" in info["kernel"], info
    _, pol = eng.download()
    reference.check("improved policy", pol)
    v0, _ = eng.download()
    reference.check("value_function before the sweep", v0)
    delta, _ = eng.sweeps(1)
    v1, _ = eng.download()
    reference.check("value_function after the sweep", v1)
    assert delta == float(np.max(np.abs(v1 - v0)))
    eng.close()


def test_k5_transition_rows_match_the_reference_slab_wise(reference):
    """64 M x 9 rows cannot be expanded at once (2 x 16 GB per action): compare slabs spread over the grid."""
    env, bins = "double_cartpole_swingup", 20
    eng = envs.make(env, bins=bins)
    eng.build_table()
    n = 160_000
    compared = 0
    for a, s0 in ((0, 0), (1, 3_200_000), (4, 13_333_337), (8, 31_999_999), (2, 50_000_000), (6, 60_500_000),
                  (7, 64_000_000 - n)):
        idx, w, r, t = eng.expand_rows(a, s0, n)
        own = t != 2                      # states in the terminal mask have no row (new_V := V, :1053)
        live = own & (t != 1)
        slab = f"action {a} states {s0}+{n}"
        reference.check(f"{slab} terminated", (t == 1)[own])
        reference.check(f"{slab} idx", idx[live])
        reference.check(f"{slab} w", w[live])
        reference.check(f"{slab} reward", r[own])
        compared += int(own.sum())
    assert compared >= 4 * n          # the first and the last slab (and the end of the sixth) lie in the terminal mask |x| > 2.4
    eng.close()


@pytest.mark.timeout(900)
def test_k5_bins12_runs_to_the_same_stable_policy_as_the_reference(reference):
    """The autoresearch trial workload (--bins 12, 2 985 984 states) with the reference's own config, to the end."""
    env, bins = "double_cartpole_swingup", 12
    eng = envs.make(env, bins=bins)
    eng.run()
    assert eng.converged
    reference.check_run(eng)
