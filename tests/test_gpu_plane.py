"""The plane-staged evaluation sweep (csrc/plane_sweep_src.cuh + csrc/plane_plan.cuh: V-planes staged in shared
memory by TMA bulk copies after a per-policy plan, corners read by LDS) must be bit-identical to the engine's
gather sweeps — and therefore to the reference's policy_eval_kernel_4d/_6d
(src/cuda_policy_iteration.py:616-649, :1044-1079) — for every policy: regular, greedy (bang-bang), random
(more successor cells per state-plane than the plan stages -> global-gather fallback), with terminated /
absorbing rows, clamped edges, wrapped angles, too few slots (late loads, unstaged cells) and ragged chunks."""
import numpy as np
import pytest

from dynamicprogramming_b200 import envs

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _prepared(env, bins, monkeypatch, layout=None, sweeps=7, policy="greedy"):
    if layout is not None:
        monkeypatch.setenv("DPB200_FAST_DIM", layout)
    monkeypatch.setenv("DPB200_PLANE", "off")    # the engine's own sweeps stay on the gather kernels: they are the comparison
    eng = envs.make(env, bins=bins)
    eng.build_table()
    if policy == "greedy":
        eng.sweeps(3)
        eng.policy_improvement()
    elif policy == "random":
        eng.upload_policy(np.random.default_rng(5).integers(0, eng.n_actions, eng.n_states).astype(np.int32))
    eng.sweeps(sweeps)
    return eng


CART = [("double_cartpole_swingup", 8), ("double_cartpole", 8), ("double_cartpole_swingup", 10), ("cartpole", 12),
        ("cartpole_swingup", 16)]


@pytest.mark.parametrize("env,bins", CART)
def test_layout_probe_finds_the_cart_plane(env, bins, monkeypatch):
    """Cart position and velocity (dims 0, 1) are the two translation-invariant dimensions of every cart-pole
    environment: the probe must store them fastest."""
    monkeypatch.setenv("DPB200_PLANE", "off")
    eng = envs.make(env, bins=bins)
    lay = eng.layout()
    if eng.N_DIMS == 6:
        assert sorted(lay["perm"][-2:]) == [0, 1], lay
    else:   # coarse 4-D grids: other pairs can tie at one successor cell per plane; a plane must have been found
        assert lay["perm"][-1] == lay["fast_dim"] and lay["fast_dim2"] >= 0, lay
    eng.close()


@pytest.mark.parametrize("env,bins", CART)
@pytest.mark.parametrize("policy", ["initial", "greedy", "random"])
@pytest.mark.parametrize("cfg", ["", "0,0,2,2,0", "0,3,1,1,1", "40,7,2,2,1", "0,0,2,2,2", "0,3,1,1,2", "40,7,2,2,2"])
def test_plane_sweep_is_bit_identical_to_the_gather_sweep(env, bins, policy, cfg, monkeypatch):
    eng = _prepared(env, bins, monkeypatch, policy=policy)
    if cfg.startswith("40") and eng.N_DIMS == 4:
        cfg = "10" + cfg[2:]     # 4-D: 4 corner planes per cell
    out = eng.debug_plane(cfg, iters=2)
    assert out["mismatches"] == 0, out
    if policy != "random":
        assert out["fallback_frac"] < 0.05, out
    eng.close()


@pytest.mark.parametrize("env,bins,layout", [("double_pendulum_swingup", 12, "0,1"), ("overhead_crane", 12, "3,2"),
                                             ("double_cartpole_swingup", 8, "5,3"), ("cartpole", 12, "2,0")])
def test_plane_sweep_without_plane_structure_falls_back_correctly(env, bins, layout, monkeypatch):
    """Forced storage orders whose planes see many successor cells: most states take the global-gather
    fallback, results must not change."""
    eng = _prepared(env, bins, monkeypatch, layout=layout)
    out = eng.debug_plane("", iters=1)
    assert out["mismatches"] == 0, out
    eng.close()


@pytest.mark.parametrize("env,bins", [("double_cartpole_swingup", 8), ("cartpole", 12), ("double_cartpole", 10)])
def test_full_policy_iteration_with_the_plane_sweep_matches_the_reference(env, bins, monkeypatch, reference):
    """Complete run() with the plane-staged sweep forced on: PI iterations, sweep counts, policy and V bits
    equal the reference's own kernels."""
    monkeypatch.setenv("DPB200_PLANE", "force")
    spec = envs.REGISTRY[env]
    c = spec.config()
    c.max_pi_iter, c.max_eval_iter = 4, 300
    eng = spec.make(bins=bins, config=c)
    eng.build_table()
    info = eng.eval_kernel_info()
    assert info["plane"] and "ps_sweep" in info["kernel"], info
    eng.run()
    reference.check_run(eng)


def test_plane_autotune_never_changes_results(monkeypatch):
    runs = {}
    for mode in ("off", "auto", "force"):
        monkeypatch.setenv("DPB200_PLANE", mode)
        spec = envs.REGISTRY["double_cartpole_swingup"]
        c = spec.config()
        c.max_pi_iter, c.max_eval_iter = 2, 120
        eng = spec.make(bins=8, config=c)
        eng.run()
        runs[mode] = (eng.policy.copy(), eng.value_function.copy(), eng.total_eval_sweeps)
    for mode in ("auto", "force"):
        assert runs[mode][2] == runs["off"][2]
        np.testing.assert_array_equal(runs[mode][0], runs["off"][0])
        np.testing.assert_array_equal(bits(runs[mode][1]), bits(runs["off"][1]))


@pytest.mark.parametrize("env,bins,plane", [("double_cartpole_swingup", 8, "force"), ("double_cartpole_swingup", 10, "force:0,3,2,2,0"),
                                            ("cartpole", 14, "force")])
def test_pipelined_policy_upload_equals_the_serial_upload(env, bins, plane, monkeypatch):
    """pi_upload_policy_local with the plane-staged sweep ready sends the slice in pieces and compacts / plans each piece
    while the next one is on the link (plan kernels over state-plane ranges): same rows, same plan, same V bits as one
    copy followed by one compaction and one plan — and as the gather sweep."""
    res = {}
    P = None
    for mode in ("serial", "pipelined", "gather"):
        monkeypatch.setenv("DPB200_PLANE", "off" if mode == "gather" else plane)
        monkeypatch.setenv("DPB200_UPLOAD", "serial" if mode == "serial" else "auto")
        eng = envs.make(env, bins=bins)
        eng.build_table()
        if mode != "gather":
            assert "ps_sweep" in eng.eval_kernel_info()["kernel"]
        eng.sweeps(5)
        if P is None:
            rng = np.random.default_rng(11)
            eng.policy_improvement()
            P = np.where(rng.random(eng.n_states) < 0.1, rng.integers(0, eng.n_actions, eng.n_states), eng.download()[1]).astype(np.int32)
        for rep in range(2):   # twice: the second upload starts while nothing of the first is pending
            eng.upload_policy_local(eng.to_internal_order(P))
            eng.sweeps(26)
        v, p = eng.download()
        res[mode] = (bits(v).copy(), p.copy())
        eng.close()
    for mode in ("pipelined", "gather"):
        np.testing.assert_array_equal(res[mode][0], res["serial"][0])
        np.testing.assert_array_equal(res[mode][1], res["serial"][1])


def test_debug_hooks_under_the_plane_sweep_leave_the_engine_as_it_was(monkeypatch):
    """debug_pair and debug_xline on an engine that runs the plane-staged sweep: they set it aside with the other JIT
    sweeps and compare their candidate with the gather sweep; afterwards the engine selects the same kernel and sweeps
    to the same V bits as a twin that never called them."""
    monkeypatch.setenv("DPB200_FAST_DIM", "0,1")   # dims 0, 1 fastest: a plane layout on which x-line sweeps apply
    monkeypatch.setenv("DPB200_PLANE", "force")
    engines = []
    for _ in range(2):
        eng = envs.make("double_cartpole_swingup", bins=8)
        eng.build_table()
        eng.sweeps(3)
        eng.policy_improvement()
        eng.sweeps(4)
        engines.append(eng)
    eng, twin = engines
    before = eng.eval_kernel_info()
    assert before["plane"] and "ps_sweep" in before["kernel"], before
    out = eng.debug_pair(128, 8, iters=1, lv=2, group=8, single=1)
    assert out["mismatches"] == 0, out
    out = eng.debug_xline("4,0,4,8,1,1:1,1,2,4,4", iters=1)
    assert out["mismatches"] == 0, out
    assert eng.eval_kernel_info() == before
    for e in engines:
        e.sweeps(5)
    np.testing.assert_array_equal(bits(eng.download()[0]), bits(twin.download()[0]))
    for e in engines:
        e.close()
