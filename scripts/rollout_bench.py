#!/usr/bin/env python3
"""Closed-loop rollout throughput on K5 (the 6-D double cart-pole swing-up): the fused rollout kernel
(pi_rollout_run: one thread per episode, lookup + step_dynamics in one kernel) with recording off and on, against
what the API allows without it — a Python loop of PolicyLookup + pi_rollout_step, two calls per step.

    python scripts/rollout_bench.py --out DIR [--episodes 65536] [--steps 1000]

Workloads: K5 at --bins 12 with the policy trained to stable, and K5 at --bins 20 with the policy after one PI
iteration.  Start states are seeded uniform draws inside the grid.  Times are host clocks around each call, which ends
in a stream synchronise; rates are episode-steps (the sum of the episodes' lengths) per second.  The Python loop is
checked to give the fused kernel's lengths and returns bit for bit.  Prints the GPU name and power limit and writes
DIR/rollout_bench.json."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
try:
    from loguru import logger

    logger.remove()
except ImportError:
    pass
import numpy as np

from dynamicprogramming_b200 import envs
from dynamicprogramming_b200.utils import PolicyLookup, PolicyRollout


def gpu_info() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return r.stdout.strip()


def timed(fn, repeat):
    ts, out = [], None
    for _ in range(repeat):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), ts, out


def python_loop(look, roll, x0, T):
    """The same episodes, one PolicyLookup call and one pi_rollout_step call per step over the live episodes."""
    n = len(x0)
    x = x0.copy()
    length = np.zeros(n, np.int32)
    term = np.zeros(n, bool)
    rew = np.zeros((n, T), np.float32)
    for t in range(T):
        alive = np.nonzero(~term)[0]
        if len(alive) == 0:
            break
        a = look(x[alive])
        nx, r, tm = roll.step(x[alive], a)
        x[alive], rew[alive, t], length[alive], term[alive] = nx, r, t + 1, tm
    return length, term, rew


def bench(name, eng, policy, gamma, n, T, repeat):
    rng = np.random.default_rng(0)
    lo, hi = eng.bounds_low, eng.bounds_high
    x0 = (lo + (hi - lo) * rng.random((n, eng.N_DIMS))).astype(np.float32)
    src = eng._dynamics_cuda_src()
    roll = PolicyRollout(policy, eng.action_space, lo, hi, eng.grid_shape, src)
    look = PolicyLookup(policy, eng.action_space, lo, hi, eng.grid_shape)
    roll.run(x0[:1024], 10, gamma, record=True)                 # warm-up: module load, workspace
    ms_off, all_off, res = timed(lambda: roll.run(x0, T, gamma), repeat)
    ms_on, all_on, rec = timed(lambda: roll.run(x0, T, gamma, record=True), repeat)
    steps = int(res.length.sum())
    t0 = time.perf_counter()
    length, term, rew = python_loop(look, roll, x0, T)
    s_loop = time.perf_counter() - t0
    total = np.zeros(n)
    for t in range(T):                                           # host float64 sum in step order
        m = t < length
        total[m] = total[m] + rew[m, t].astype(np.float64)
    match = bool(np.array_equal(length, res.length) and np.array_equal(term, res.terminated)
                 and np.array_equal(total.view(np.uint64), res.total_reward.view(np.uint64))
                 and np.array_equal(rec.total_reward.view(np.uint64), res.total_reward.view(np.uint64)))
    roll.close()
    look.close()
    row = {"workload": name, "episodes": n, "steps": T, "episode_steps": steps, "gamma": gamma,
           "mean_length": float(res.length.mean()), "terminated": float(res.terminated.mean()),
           "mean_return": float(res.total_reward.mean()), "mean_discounted_return": float(res.discounted_return.mean()),
           "fused_s": ms_off, "fused_s_all": all_off, "fused_steps_per_s": steps / ms_off,
           "fused_record_s": ms_on, "fused_record_s_all": all_on, "fused_record_steps_per_s": steps / ms_on,
           "python_loop_s": s_loop, "python_loop_steps_per_s": steps / s_loop, "loop_matches_fused": match}
    print(json.dumps(row), flush=True)
    return row


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--episodes", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--out", type=Path, required=True, help="directory for rollout_bench.json")
    args = ap.parse_args()
    info = gpu_info()
    print(info, flush=True)
    spec = envs.REGISTRY["double_cartpole_swingup"]
    gamma = float(np.float32(spec.config().gamma))
    rows = []

    t0 = time.perf_counter()
    eng = envs.make("double_cartpole_swingup", bins=12)
    eng.run()
    print(f"K5 bins 12: {eng.pi_iterations} PI iterations, converged={eng.converged}, {time.perf_counter() - t0:.1f} s",
          flush=True)
    rows.append(bench("K5 bins 12, stable policy", eng, eng.policy, gamma, args.episodes, args.steps, args.repeat))

    t0 = time.perf_counter()
    eng = envs.make("double_cartpole_swingup", bins=20)
    eng.policy_evaluation()
    eng.policy_improvement()
    _, policy = eng.download()
    eng.close()
    print(f"K5 bins 20: policy after one PI iteration, {time.perf_counter() - t0:.1f} s", flush=True)
    rows.append(bench("K5 bins 20, policy after one PI iteration", eng, policy, gamma, args.episodes, args.steps,
                      args.repeat))

    args.out.mkdir(parents=True, exist_ok=True)
    (args.out / "rollout_bench.json").write_text(json.dumps({"gpu": info, "rows": rows}, indent=1))
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
