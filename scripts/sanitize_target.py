#!/usr/bin/env python3
"""One sweep family on a small grid, for compute-sanitizer (tests/test_gpu_sanitizer.py):
    compute-sanitizer --tool memcheck --error-exitcode 1 python scripts/sanitize_target.py <family>
families: aot | gp_single | gp_pair | xline | persistent | plane | plane_small | plane_scalar | plane_items_small | lookup |
          rollout | odd_aot5 | odd_xline3 | odd_plane5 | warm_start
warm_start prolongs a coarser and a finer source value function onto an engine with a terminal mask (the overhead
crane, whose goal states also carry values from set_values) and runs an improvement and sweeps from it.
The odd_* families run the chain-of-integrators fixture of tests/fixtures/odd_dims.py at D = 3 or 5 (rows with an odd
number of words)."""
import importlib.util
import os
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
family = sys.argv[1]
env, bins = "double_cartpole_swingup", 6
cfg = {
    "aot": {"DPB200_PLANE": "off", "DPB200_XLINE": "off", "DPB200_PAIR": "off"},
    "gp_single": {"DPB200_PLANE": "off", "DPB200_XLINE": "off", "DPB200_PAIR": "force:128,8,2,8,1"},
    "gp_pair": {"DPB200_PLANE": "off", "DPB200_XLINE": "off", "DPB200_PAIR": "force:64,8,2,8,0"},
    "xline": {"DPB200_PLANE": "off", "DPB200_FAST_DIM": "0", "DPB200_XLINE": "force:2,0,4,8,2,1:1,1,1,2,6"},
    "persistent": {"DPB200_PLANE": "off", "DPB200_XLINE": "off", "DPB200_PAIR": "off", "DPB200_PERSIST": "on"},
    "plane": {"DPB200_PLANE": "force"},
    "plane_small": {"DPB200_PLANE": "force:34,5,2,1,1"},
    "plane_scalar": {"DPB200_PLANE": "force:0,0,2,2,0"},
    "plane_items_small": {"DPB200_PLANE": "force:34,5,2,2,2"},
    "lookup": {},
    "rollout": {},
    "odd_aot5": {"DPB200_PLANE": "off", "DPB200_XLINE": "off", "DPB200_PAIR": "off"},
    "odd_xline3": {"DPB200_PLANE": "off", "DPB200_FAST_DIM": "0", "DPB200_XLINE": "force:2,0,4,8,2,1:1,1"},
    "odd_plane5": {"DPB200_FAST_DIM": "0,1", "DPB200_PLANE": "force:0,0,2,2,2"},
    "warm_start": {},
}[family]
os.environ.update(cfg)
os.environ["DPB200_CACHE"] = "off"
if family == "persistent":
    env, bins = "cartpole", 10
if family == "warm_start":
    env, bins = "overhead_crane", 11
import numpy as np

from dynamicprogramming_b200 import envs

if family.startswith("odd_"):
    spec = importlib.util.spec_from_file_location("odd_dims", ROOT / "tests" / "fixtures" / "odd_dims.py")
    odd = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(odd)
    eng = odd.make(int(family[-1]))
else:
    eng = envs.make(env, bins=bins)
eng.build_table()
info = eng.eval_kernel_info()["kernel"]
want = {"aot": "eval_sweep_kernel", "gp_single": "gp_sweep", "gp_pair": "gp_sweep", "xline": "xl_sweep",
        "persistent": "eval_persistent_kernel", "plane": "ps_sweep", "plane_small": "ps_sweep", "plane_scalar": "ps_sweep", "plane_items_small": "ps_sweep", "lookup": "", "rollout": "",
        "odd_aot5": "eval_sweep_kernel<5>", "odd_xline3": "xl_sweep", "odd_plane5": "ps_sweep",
        "warm_start": ""}[family]
assert want in info, (family, info)
eng.sweeps(3)
eng.policy_improvement()
d, _ = eng.sweeps(26)                 # a whole sync interval + a check sweep
eng.upload_policy(np.random.default_rng(1).integers(0, eng.n_actions, eng.n_states).astype(np.int32))
eng.sweeps(2)
if family == "lookup":
    pts = np.random.default_rng(2).uniform(-1, 1, (257, eng.N_DIMS)).astype(np.float32)
    eng.lookup_actions(pts)
if family == "rollout":   # pi_rollout_episodes, pi_step_states and the shared-memory tiles of rollout_unstage_kernel
    rng = np.random.default_rng(3)
    lo, hi = eng.bounds_low, eng.bounds_high
    x0 = (lo + (hi - lo) * rng.uniform(-0.1, 1.1, (333, eng.N_DIMS))).astype(np.float32)
    res = eng.rollout(x0, 37, record=True)
    assert res.states.shape == (333, 38, eng.N_DIMS) and (res.length >= 1).all()
    eng.simulate_step(x0, np.full(len(x0), eng.action_space[0], np.float32))
if family == "warm_start":   # pi_prolong_values from a coarser and a finer source, then improvement + sweeps
    for b in (7, 16):
        n = b ** eng.N_DIMS
        src = np.random.default_rng(b).standard_normal(n).astype(np.float32)
        eng.warm_start((src, eng.bounds_low, eng.bounds_high, np.full(eng.N_DIMS, b)))
        eng.sweeps(3)
v, p = eng.download()
assert np.isfinite(v).all()
eng.close()
print("SANITIZE_TARGET_OK", family, info[:60])
