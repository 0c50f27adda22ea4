"""The x-line evaluation sweep (csrc/xline_sweep_src.cuh: vector window loads, packed fp32
arithmetic, tile-ordered rows, JIT-compiled per grid) must be bit-identical to the scalar
gather sweep — and therefore to the reference's policy_eval_kernel_4d/_6d
(src/cuda_policy_iteration.py:616-649, :1044-1079) — on every environment, including the
ones whose successors are NOT consecutive along the fast dimension (scalar fallback path),
terminated / absorbing rows, clamped edges and wrapped angles."""
import numpy as np
import pytest

from dynamicprogramming_b200 import envs

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _prepared(env, bins, monkeypatch, sweeps=7):
    monkeypatch.setenv("DPB200_FAST_DIM", "0")   # the x-line sweep needs logical dimension 0 stored fastest
    monkeypatch.setenv("DPB200_XLINE", "off")    # the engine's own sweeps stay scalar: they are the comparison
    eng = envs.make(env, bins=bins)
    eng.build_table()
    eng.policy_improvement()
    eng.sweeps(sweeps)
    return eng


CASES_6D = [("double_cartpole_swingup", 8), ("double_cartpole", 8)]
CASES_4D = [("cartpole", 12), ("cartpole_swingup", 16), ("double_pendulum_swingup", 12), ("overhead_crane", 12)]


@pytest.mark.parametrize("env,bins", CASES_6D + CASES_4D)
@pytest.mark.parametrize("cfg", ["2,0,4,8,2,1", "4,0,4,8,1,1", "4,0,2,4,1,2", "2,1,2,4,2,4", "4,1,4,8,1,1"])
def test_xline_sweep_is_bit_identical_to_the_scalar_sweep(env, bins, cfg, monkeypatch):
    eng = _prepared(env, bins, monkeypatch)
    D = eng.N_DIMS
    K, warps = int(cfg.split(",")[0]), int(cfg.split(",")[3])
    # tile: fill the CTA's x-line slots from the fastest non-fast position
    slots, tile = warps * (32 // (bins // K)), [1] * (D - 1)
    for k in range(D - 2, -1, -1):
        t = max(d for d in range(1, bins + 1) if bins % d == 0 and d <= slots)
        tile[k] = t
        slots //= t
    out = eng.debug_xline(cfg + ":" + ",".join(map(str, tile)), iters=1)
    assert out["mismatches"] == 0, out
    eng.close()


@pytest.mark.parametrize("env,bins,cfg", [("double_cartpole_swingup", 8, "force:4,0,4,8,1,1:1,1,2,4,4"),
                                          ("cartpole", 12, "force:2,0,4,8,2,1:1,3,6"),
                                          ("double_pendulum_swingup", 12, "force:4,0,4,8,1,1:2,4,6")])
def test_full_policy_iteration_with_the_xline_sweep_matches_the_reference(env, bins, cfg, monkeypatch, reference):
    """Complete run() with the x-line sweep forced on: PI iterations, sweep counts, policy and V bits
    equal the reference's own kernels."""
    monkeypatch.setenv("DPB200_FAST_DIM", "0")
    monkeypatch.setenv("DPB200_XLINE", cfg)
    spec = envs.REGISTRY[env]
    c = spec.config()
    c.max_pi_iter, c.max_eval_iter = 4, 300
    eng = spec.make(bins=bins, config=c)
    eng.build_table()
    info = eng.eval_kernel_info()
    assert info["xline"], info
    eng.run()
    reference.check_run(eng)


def test_autotune_reports_its_choice_and_never_changes_results(monkeypatch):
    runs = {}
    for mode in ("off", "auto"):
        monkeypatch.setenv("DPB200_XLINE", mode)
        spec = envs.REGISTRY["double_cartpole_swingup"]
        c = spec.config()
        c.max_pi_iter, c.max_eval_iter = 2, 120
        eng = spec.make(bins=8, config=c)
        eng.build_table()
        info = eng.eval_kernel_info()   # before run(): run() releases the device side like the reference
        assert info["kernel"] and (mode == "auto" or not info["xline"])
        eng.run()
        runs[mode] = (eng.total_eval_sweeps, eng.policy.copy(), bits(eng.value_function).copy())
        eng.close()
    assert runs["off"][0] == runs["auto"][0]
    np.testing.assert_array_equal(runs["off"][1], runs["auto"][1])
    np.testing.assert_array_equal(runs["off"][2], runs["auto"][2])


def test_upload_policy_refreshes_the_tile_ordered_rows(monkeypatch):
    """pi_upload_policy re-compacts AND re-tiles: sweeps after an upload use the new policy's rows."""
    monkeypatch.setenv("DPB200_FAST_DIM", "0")
    res = {}
    for mode in ("off", "force:2,0,4,8,2,1:1,1,1,2,4"):
        monkeypatch.setenv("DPB200_XLINE", mode)
        eng = envs.make("double_cartpole_swingup", bins=8)
        eng.build_table()
        rng = np.random.default_rng(5)
        eng.upload_policy(rng.integers(0, eng.n_actions, eng.n_states).astype(np.int32))
        eng.sweeps(5)
        v = np.empty(eng.n_states, np.float32)
        eng.download(values=v)
        res[mode] = bits(v).copy()
        eng.close()
    a, b = res.values()
    np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize("env,bins", [("double_cartpole_swingup", 8), ("cartpole_swingup", 16), ("double_pendulum_swingup", 13),
                                      ("overhead_crane", 11)])
def test_packed_pair_sweep_is_bit_identical_to_the_scalar_sweep(env, bins, monkeypatch):
    """csrc/pair_sweep_src.cuh (two states per thread, FMUL2/FFMA2, immediate gather offsets; any storage order,
    odd sizes) against pi::eval_sweep_kernel, then a full run with it forced on against the reference kernels."""
    monkeypatch.setenv("DPB200_XLINE", "off")
    monkeypatch.setenv("DPB200_PAIR", "off")
    eng = envs.make(env, bins=bins)
    eng.build_table()
    eng.sweeps(20)
    eng.policy_improvement()
    eng.sweeps(5)
    for threads, minb in ((64, 8), (256, 2)):
        out = eng.debug_pair(threads, minb, iters=1)
        assert out["mismatches"] == 0, out
    # lean weight-tree levels and explicitly scheduled gather groups, packed pairs and ONE state per thread
    # (the default generic sweep of large 6-D grids: 128 x 8, lv 2, groups of 8)
    for threads, minb, lv, group, single in ((64, 8, 2, 8, False), (128, 4, 3, 16, False), (128, 8, 2, 8, True),
                                             (128, 8, 1, 0, True), (256, 4, 3, 4, True), (128, 16, 1, 0, True),
                                             (64, 16, 2, 16, True)):
        out = eng.debug_pair(threads, minb, iters=1, lv=lv, group=group, single=single)
        assert out["mismatches"] == 0, (threads, minb, lv, group, single, out)
    # pair-shadow gathers (P[i] = (V[i], V[i+1]), one 64-bit load per cell edge along the fast dimension): needs
    # logical dimension 0 stored fastest
    if eng.layout()["fast_dim"] == 0:
        for group in (2, 8, 16):
            out = eng.debug_pair(128, 8, iters=2, lv=2, group=group, single=2)
            assert out["mismatches"] == 0, (group, out)
    eng.close()


@pytest.mark.parametrize("variant", [2, 12, 44, 64, 128, 192, 256])
def test_scalar_sweep_tuning_variants_are_bit_identical(variant, monkeypatch):
    """DPB200_EVAL_VARIANT (L2 eviction policies, forced occupancy, lean weight tree, explicitly grouped gathers):
    same V bits as the default scalar sweep on a 6-D and a 4-D environment."""
    monkeypatch.setenv("DPB200_XLINE", "off")
    monkeypatch.setenv("DPB200_PAIR", "off")
    for env, bins in (("double_cartpole_swingup", 7), ("cartpole_swingup", 15)):
        res = []
        for var in (0, variant):
            monkeypatch.setenv("DPB200_EVAL_VARIANT", str(var))
            eng = envs.make(env, bins=bins)
            eng.build_table()
            eng.sweeps(20)
            eng.policy_improvement()
            eng.sweeps(7)
            v, _ = eng.download()
            res.append(bits(v).copy())
            eng.close()
        np.testing.assert_array_equal(res[0], res[1])


def test_full_policy_iteration_with_the_single_state_jit_sweep_matches_the_reference(monkeypatch, reference):
    monkeypatch.setenv("DPB200_XLINE", "off")
    monkeypatch.setenv("DPB200_PAIR", "force:128,8,2,8,1")
    for env, bins in (("double_cartpole_swingup", 6), ("cartpole", 12)):
        spec = envs.REGISTRY[env]
        c = spec.config()
        c.max_pi_iter, c.max_eval_iter = 3, 200
        eng = spec.make(bins=bins, config=c)
        eng.build_table()
        assert "one state/thread" in eng.eval_kernel_info()["kernel"]
        eng.run()
        reference.check_run(eng, f"{env} ")


def test_full_policy_iteration_with_the_packed_pair_sweep_matches_the_reference(monkeypatch, reference):
    monkeypatch.setenv("DPB200_XLINE", "off")
    monkeypatch.setenv("DPB200_PAIR", "force")
    spec = envs.REGISTRY["double_cartpole"]
    c = spec.config()
    c.max_pi_iter, c.max_eval_iter = 3, 200
    eng = spec.make(bins=7, config=c)
    eng.build_table()
    assert "gp_sweep" in eng.eval_kernel_info()["kernel"]
    eng.run()
    reference.check_run(eng)
