#!/usr/bin/env python3
"""Recompute mode against full-table mode (DPB200_TABLE, include/dpb200.h: pi_create), and a grid whose table does not fit.

    python scripts/recompute_bench.py --out DIR [--repeats 1] [--big-bins 30] [--skip-small] [--skip-big]

1. K5 (double_cartpole_swingup --bins 20, the runner's config): run() to a stable policy in `full` and in `recompute`
   mode, alternated in one process (`--repeats` pairs).  Per run: wall time of the table build and of run(), the
   engine's device timings (build_ms, improve_ms per pass, eval_ms per sweep), PI iterations, sweeps, and whether the
   policy and the V bits equal the first full-mode run's.
2. K5 at --bins 30 under DPB200_TABLE=auto: the mode the engine chose, the device memory in use after the build
   (cudaMemGetInfo), the build time, and a capped solve (2 PI iterations x 200 sweeps), cold and warm-started from the
   --bins 20 solution of part 1: per PI iteration the evaluation and improvement device times and the ms per sweep.
Wall times are host clocks around calls that end in a stream synchronise; device times are the engine's CUDA events.
Prints the GPU name and power limit and writes DIR/recompute_bench.json."""
import argparse
import json
import os
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

ENV = "double_cartpole_swingup"


def gpu_info() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip()


def used_gb() -> float:
    import torch

    free, total = torch.cuda.mem_get_info()
    return (total - free) / 1e9


def run_small(spec, mode, bins):
    os.environ["DPB200_TABLE"] = mode
    t0 = time.perf_counter()
    pi = spec.make(bins=bins)
    pi.build_table()
    build_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    pi.run()
    run_s = time.perf_counter() - t0
    st = pi.stats
    row = {"mode": st["table_mode"], "build_wall_s": build_s, "run_wall_s": run_s, "total_wall_s": build_s + run_s,
           "build_ms": st["build_ms"], "improve_ms_per_pass": st["improve_ms"] / max(1, pi.pi_iterations),
           "eval_ms_per_sweep": st["eval_ms"] / max(1, st["eval_sweeps"]), "pi_iterations": pi.pi_iterations,
           "sweeps": pi.total_eval_sweeps, "converged": bool(pi.converged), "table_bytes": st["table_bytes"]}
    return pi, row


def capped(spec, bins, source, n_pi, n_sweeps):
    os.environ["DPB200_TABLE"] = "auto"
    cfg = spec.config()
    cfg.max_eval_iter, cfg.max_pi_iter = n_sweeps, n_pi
    t0 = time.perf_counter()
    pi = spec.make(bins=bins, config=cfg)
    pi.build_table()
    row = {"build_wall_s": time.perf_counter() - t0, "n_states": pi.n_states}
    st = pi.engine_stats()
    row.update(mode=st["table_mode"], table_bytes=st["table_bytes"], build_ms=st["build_ms"], used_gb_after_build=used_gb())
    if source is not None:
        t0 = time.perf_counter()
        ws = pi.warm_start(source)
        row["warm_start_wall_s"] = time.perf_counter() - t0
        row["warm_start_changed"] = ws["changed"]
    iters = []
    t_solve = time.perf_counter()
    for _ in range(n_pi):
        a = pi.engine_stats()
        delta = pi.policy_evaluation()
        stable = pi.policy_improvement()
        b = pi.engine_stats()
        sweeps = b["eval_sweeps"] - a["eval_sweeps"]
        iters.append({"sweeps": sweeps, "delta": delta, "changed": pi.last_changed, "stable": stable,
                      "eval_ms": b["eval_ms"] - a["eval_ms"], "ms_per_sweep": (b["eval_ms"] - a["eval_ms"]) / max(1, sweeps),
                      "improve_ms": b["improve_ms"] - a["improve_ms"]})
    row["solve_wall_s"] = time.perf_counter() - t_solve
    row["used_gb_peak_observed"] = used_gb()
    row["iterations"] = iters
    pi.close()
    return row


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", type=Path, required=True)
    ap.add_argument("--bins", type=int, default=20)
    ap.add_argument("--big-bins", type=int, default=30)
    ap.add_argument("--repeats", type=int, default=1, help="full / recompute pairs at --bins")
    ap.add_argument("--capped-pi", type=int, default=2)
    ap.add_argument("--capped-sweeps", type=int, default=200)
    ap.add_argument("--skip-small", action="store_true")
    ap.add_argument("--skip-big", action="store_true")
    args = ap.parse_args()
    args.out.mkdir(parents=True, exist_ok=True)
    gpu = gpu_info()
    print("GPU (name, power limit):", gpu, flush=True)
    spec = envs.REGISTRY[ENV]
    result = {"gpu": gpu, "env": ENV, "timing": "wall: host clock around calls ending in a stream synchronise; *_ms: the "
                                                  "engine's CUDA events", "small": [], "big": []}
    out = args.out / "recompute_bench.json"
    source = None
    if not args.skip_small:
        ref = None
        for r in range(args.repeats):
            for mode in ("full", "recompute"):
                pi, row = run_small(spec, mode, args.bins)
                if ref is None:
                    ref = (pi.policy.copy(), pi.value_function.view(np.uint32).copy())
                    source = pi
                row["repeat"] = r
                row["policy_equal"] = bool(np.array_equal(pi.policy, ref[0]))
                row["v_bits_equal"] = bool(np.array_equal(pi.value_function.view(np.uint32), ref[1]))
                result["small"].append(row)
                print(json.dumps(row), flush=True)
                out.write_text(json.dumps(result, indent=1))
        by = {m: [r for r in result["small"] if r["mode"] == m] for m in ("full", "recompute")}
        if by["full"] and by["recompute"]:
            mean = lambda rows, k: sum(r[k] for r in rows) / len(rows)
            result["small_summary"] = {
                "recompute_minus_full_total_wall_s": mean(by["recompute"], "total_wall_s") - mean(by["full"], "total_wall_s"),
                "improve_ms_per_pass": {m: mean(by[m], "improve_ms_per_pass") for m in by},
                "build_ms": {m: mean(by[m], "build_ms") for m in by},
                "all_equal": all(r["policy_equal"] and r["v_bits_equal"] for r in result["small"])}
            print(json.dumps(result["small_summary"]), flush=True)
    if not args.skip_big:
        for src in (None, source) if source is not None else (None,):
            row = capped(spec, args.big_bins, src, args.capped_pi, args.capped_sweeps)
            row["start"] = "cold" if src is None else f"warm from --bins {args.bins}"
            result["big"].append(row)
            print(json.dumps(row), flush=True)
            out.write_text(json.dumps(result, indent=1))
    out.write_text(json.dumps(result, indent=1))
    print("wrote", out)
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
