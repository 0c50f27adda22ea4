#!/usr/bin/env python3
"""Warm start against cold start to a stable policy (engine.warm_start, include/dpb200.h: pi_prolong_values).

    python scripts/warm_start_bench.py --out DIR [--cases K5,K4,K1] [--extra-coarse] [--episodes 4096] [--steps 1000]

Cases: K5 (double_cartpole_swingup --bins 20) warm from --bins 12 (and from 10 and 15 with --extra-coarse), K4
(double_pendulum_swingup --bins 50) from 25, K1 (pendulum --bins 200) from 100, each with the runner's config.
Per case: the cold solve (construct, table build, run()), the coarse solve (construct + run()), and the warm solve
(construct, table build, warm_start() = prolongation + one improvement, run()).  Wall times are host clocks around
each call, all of which end in a stream synchronise; the prolongation kernel's device time is CUDA events
(pi_prolong_values).  Also: PI iterations and evaluation sweeps of each solve, max |V_warm - V_cold|, the fraction of
states with the same action, and the closed-loop mean return of both final policies over the same seeded start states
(engine.rollout, the plugin's own dynamics, the runner's gamma).  Prints the GPU name and power limit and writes
DIR/warm_start_bench.json."""
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

from dynamicprogramming_b200 import envs, runners

CASES = {"K5": ("double_cartpole_swingup", 20, [12]), "K4": ("double_pendulum_swingup", 50, [25]),
         "K1": ("pendulum", 200, [100])}


def gpu_info() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip()


def clock(fn):
    t0 = time.perf_counter()
    out = fn()
    return time.perf_counter() - t0, out


def solve(spec, bins, source=None):
    """(engine after run(), times): construct, table build, warm start (if any), run()."""
    t = {}
    t["construct_s"], pi = clock(lambda: spec.make(bins=bins))
    t["build_s"], _ = clock(pi.build_table)
    if source is not None:
        t["warm_start_s"], ws = clock(lambda: pi.warm_start(source))
        t["prolong_device_ms"] = ws["prolong_ms"]
        t["warm_start_changed"] = ws["changed"]
    t["run_s"], _ = clock(pi.run)
    t["total_s"] = sum(v for k, v in t.items() if k.endswith("_s"))
    t.update(pi_iterations=pi.pi_iterations, sweeps=pi.total_eval_sweeps, converged=bool(pi.converged))
    return pi, t


def closed_loop(pi, spec, episodes, steps):
    gamma = float(np.float32(spec.config().gamma))
    r = pi.rollout(runners.start_states(pi, episodes, 0), steps, gamma=gamma)
    return {"mean_return": float(r.total_reward.mean()), "mean_discounted_return": float(r.discounted_return.mean()),
            "mean_length": float(r.length.mean()), "terminated": float(r.terminated.mean())}


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", type=Path, required=True)
    ap.add_argument("--cases", default="K5,K4,K1")
    ap.add_argument("--extra-coarse", action="store_true", help="K5 also from --bins 10 and 15")
    ap.add_argument("--episodes", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=1000)
    args = ap.parse_args()
    args.out.mkdir(parents=True, exist_ok=True)
    gpu = gpu_info()
    print("GPU (name, power limit):", gpu, flush=True)
    result = {"gpu": gpu, "timing": "host clock around each call (each ends in a stream synchronise); "
                                     "prolong_device_ms: CUDA events around the prolongation kernel",
              "episodes": args.episodes, "steps": args.steps, "cases": []}
    for case in args.cases.split(","):
        env, bins, coarse_list = CASES[case]
        if case == "K5" and args.extra_coarse:
            coarse_list = [12, 10, 15]
        spec = envs.REGISTRY[env]
        cold, tc = solve(spec, bins)
        cold_loop = closed_loop(cold, spec, args.episodes, args.steps)
        print(f"{case} cold bins {bins}: {json.dumps(tc)}", flush=True)
        for cb in coarse_list:
            coarse, tcr = solve(spec, cb)
            warm, tw = solve(spec, bins, coarse)
            dv = np.abs(warm.value_function.astype(np.float64) - cold.value_function.astype(np.float64))
            row = {"case": case, "env": env, "bins": bins, "coarse_bins": cb, "cold": tc, "coarse": tcr, "warm": tw,
                   "warm_total_incl_coarse_s": tcr["total_s"] + tw["total_s"],
                   "fine_sweeps_saved": tc["sweeps"] - tw["sweeps"],
                   "max_abs_dV": float(dv.max()), "V_range_cold": [float(cold.value_function.min()),
                                                                   float(cold.value_function.max())],
                   "same_action_fraction": float(np.mean(warm.policy == cold.policy)),
                   "closed_loop_cold": cold_loop, "closed_loop_warm": closed_loop(warm, spec, args.episodes, args.steps)}
            result["cases"].append(row)
            print(json.dumps(row), flush=True)
            (args.out / "warm_start_bench.json").write_text(json.dumps(result, indent=1))
    print("wrote", args.out / "warm_start_bench.json")
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
