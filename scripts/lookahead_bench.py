#!/usr/bin/env python3
"""Closed-loop rollouts under the two controllers (N8): the interpolated grid policy (pi_rollout_run) and the one-step
lookahead on the value function (pi_rollout_run_lookahead), from the same seeded starts, plus the rate of the batch
lookahead query (pi_rollout_lookahead).

    python scripts/lookahead_bench.py --out DIR [--episodes 65536] [--steps 1000] [--points 1000000]

Workloads: K5 (double cart-pole swing-up) at --bins 12, K1 (pendulum) and K3 (cart-pole) at their default bins, each
solved with run() (K5 to a stable policy; K1 and K3 to wherever their config stops).  Each controller runs --episodes
episodes of up to --steps steps from seeded uniform starts inside the grid, discounted with the runner's gamma.  Call
times are host clocks around each call, which ends in a stream synchronise (so they include the host<->device copies);
the median of --repeat calls is reported.  Rates are episode-steps (the sum of the episodes' lengths) per second and
query points per second.  Prints the GPU name and power limit and writes DIR/lookahead_bench.json."""
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
from dynamicprogramming_b200.utils import PolicyRollout

WORKLOADS = (("K5", "double_cartpole_swingup", 12), ("K1", "pendulum", None), ("K3", "cartpole", None))


def gpu_info() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip()


def timed(fn, repeat):
    ts, out = [], None
    for _ in range(repeat):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), ts, out


def bench(label, eng, gamma, n, T, n_points, repeat):
    rng = np.random.default_rng(0)
    lo, hi = eng.bounds_low, eng.bounds_high
    x0 = (lo + (hi - lo) * rng.random((n, eng.N_DIMS))).astype(np.float32)
    pts = (lo + (hi - lo) * rng.random((n_points, eng.N_DIMS))).astype(np.float32)
    roll = PolicyRollout(eng.policy, eng.action_space, lo, hi, eng.grid_shape, eng._dynamics_cuda_src())
    roll.set_values(eng.value_function)
    rows = []
    for controller in ("policy", "lookahead"):
        roll.run(x0[:1024], 10, gamma, controller=controller)          # warm-up: module load, workspace
        s, all_s, res = timed(lambda: roll.run(x0, T, gamma, controller=controller), repeat)
        steps = int(res.length.sum())
        row = {"workload": label, "controller": controller, "episodes": n, "steps": T, "gamma": gamma,
               "call_s": s, "call_s_all": all_s, "episode_steps": steps, "episode_steps_per_s": steps / s,
               "mean_return": float(res.total_reward.mean()),
               "mean_discounted_return": float(res.discounted_return.mean()),
               "mean_length": float(res.length.mean()), "terminated": float(res.terminated.mean())}
        print(json.dumps(row), flush=True)
        rows.append(row)
    roll.lookahead(pts[:1024], gamma)
    s, all_s, _ = timed(lambda: roll.lookahead(pts, gamma), repeat)
    sq, all_sq, _ = timed(lambda: roll.lookahead(pts, gamma, q=True), repeat)
    row = {"workload": label, "query_points": n_points, "actions": len(eng.action_space), "query_s": s,
           "query_s_all": all_s, "query_points_per_s": n_points / s, "query_with_q_s": sq, "query_with_q_s_all": all_sq,
           "query_with_q_points_per_s": n_points / sq}
    print(json.dumps(row), flush=True)
    rows.append(row)
    roll.close()
    return rows


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--episodes", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--points", type=int, default=1_000_000)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--out", type=Path, required=True, help="directory for lookahead_bench.json")
    args = ap.parse_args()
    info = gpu_info()
    print("GPU (name, power limit):", info, flush=True)
    rows, solves = [], []
    for key, name, bins in WORKLOADS:
        spec = envs.REGISTRY[name]
        gamma = float(np.float32(spec.config().gamma))
        t0 = time.perf_counter()
        eng = envs.make(name, bins=bins)
        eng.run()
        solve = {"workload": key, "env": name, "bins": int(eng.grid_shape[0]), "pi_iterations": eng.pi_iterations,
                 "converged": bool(eng.converged), "solve_s": time.perf_counter() - t0}
        print(json.dumps(solve), flush=True)
        solves.append(solve)
        rows += bench(f"{key} ({name}, bins {solve['bins']})", eng, gamma, args.episodes, args.steps, args.points,
                      args.repeat)
    args.out.mkdir(parents=True, exist_ok=True)
    (args.out / "lookahead_bench.json").write_text(json.dumps({"gpu": info, "solves": solves, "rows": rows}, indent=1))
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
