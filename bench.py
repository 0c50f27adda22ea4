#!/usr/bin/env python3
"""
bench.py — policy-evaluation throughput (Bellman state-backups/s) on the
reference's largest configuration: Double CartPole swing-up, 6-D, --bins 20
(64 M states, 9 actions; BASELINE.json configs[4], SURVEY.md §8 K5).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A *step* is one sync interval of the reference's policy_evaluation loop
(src/cuda_policy_iteration.py:300-336): 25 Jacobi sweeps over the whole grid
under the policy produced by the first improvement pass.  Timed with CUDA
events on the engine's stream (max over ranks).  Rank 0 prints ONE JSON line.

  value        whole-job state-backups/s with the transition rows and V resident in HBM
  e2e          the same through the public Python API with HOST buffers: every
               step uploads the policy (pinned host -> device), re-compacts the
               rows, runs the 25 sweeps and downloads V + the residual
  roofline     HBM roofline of the evaluation-sweep kernel (algorithmic bytes =
               compact row + V read + V write per backup; DESIGN.md §4)
  cpu_baseline the CPU restatement (oracle/pi_oracle.c, OpenMP) on a bounded slab
  --impl reference   the reference's OWN kernels (oracle/_ref cubins compiled by
               oracle/build_ref.py with NVRTC) driven by the reference's host loop on one
               B200 — the reference has no CPU policy-iteration path (SURVEY §8c)
  --dump-outputs DIR   after the timed steps, what the last one computed (see dump_outputs)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
# stdout carries exactly ONE JSON line: NCCL's own messages (e.g. "NCCL version ..." when the box sets
# NCCL_DEBUG) go to stderr instead of stdout
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

ENV = "double_cartpole_swingup"
SWEEPS_PER_STEP = 25
METRIC = "bellman_state_backups_per_s"
UNIT = "backups/s"


def workload_config(bins: int, n_actions: int, gamma: float, sharding: str) -> dict:
    """`config` of the JSON line — the same keys and (at N = 1) the same values in both arms."""
    N = bins ** 6
    return {"workload": f"{ENV} 6-D --bins {bins} ({N:,} states x {n_actions} actions), "
                        f"policy evaluation, step = {SWEEPS_PER_STEP} Jacobi sweeps (one reference sync interval)",
            "policy": "greedy policy after PI iteration 1", "gamma": gamma, "sharding": sharding,
            "l2": "inputs larger than L2 (rows %.2f GB + V %.2f GB per sweep)" % (8 * 4 * N / 1e9, 4 * N / 1e9)}


def v_checksum(t) -> int:
    """Order-independent 64-bit checksum of a float32 device tensor: sum of its words as unsigned integers
    (reduced on the device).  Equal checksums in both arms / at every N <=> the same multiset of V bits."""
    import torch

    return int((t.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF).sum().item())


DUMP_SAMPLE = 1 << 22   # states of V written by --dump-outputs: 16 MB of values + 32 MB of indices


def dump_outputs(out_dir: str, values: np.ndarray, residual: float) -> None:
    """What a caller of the timed path receives after its last step: V in reference order (every state up to
    DUMP_SAMPLE states, else a fixed sample drawn with seed 0, sorted) with the flat state index of each value, and
    the residual max|V_new - V_old| of the step's last sweep.  The inputs are the same in every run with the same
    arguments, so two builds can be compared file by file."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    n = values.size
    idx = np.arange(n) if n <= DUMP_SAMPLE else np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE, replace=False))
    np.save(d / "value_function.npy", values[idx].astype(np.float32))
    np.save(d / "value_function_index.npy", idx.astype(np.float64))
    np.save(d / "residual.npy", np.array([residual], dtype=np.float32))


def _quiet_logs() -> None:
    try:
        from loguru import logger

        logger.remove()
        logger.add(sys.stderr, level="WARNING")
    except ImportError:
        pass


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int) -> None:
        self.index, self.samples, self.proc = index, [], None

    def start(self) -> None:
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self) -> None:
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            parts = [p.strip() for p in s.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); pw.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak() -> tuple[float, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(bins: int) -> float | None:
    """dram bytes per evaluation-sweep launch from the committed ncu summary (profiles/)."""
    p = ROOT / "profiles" / "traffic.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get(f"{ENV}@{bins}", {}).get("eval_sweep_dram_bytes_per_launch")
        except Exception:  # noqa: BLE001
            return None
    return None


# --------------------------------------------------------------------------- ours
def run_ours(args) -> dict:
    import torch

    from dynamicprogramming_b200 import _ffi, dist as pdist, envs

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    shard = pdist.make_shard(local) if world > 1 else None
    td = pdist.init_process_group() if world > 1 else None

    spec = envs.REGISTRY[ENV]
    eng = spec.make(bins=args.bins, device=local, shard=shard)
    N = eng.n_states
    lib = _ffi.lib()
    lo, hi = lib.pi_local_begin(eng._engine), lib.pi_local_end(eng._engine)
    eng.build_table()
    # policy of PI iteration 1: a bounded evaluation of the initial policy, then one improvement
    eng.sweeps(2 * SWEEPS_PER_STEP)
    eng.policy_improvement()
    build_ms = eng.engine_stats()["build_ms"]
    improve_ms = eng.engine_stats()["improve_ms"]

    def barrier():
        torch.cuda.synchronize()
        if td is not None:
            td.barrier()

    # ---- device-resident arm -------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        eng.sweeps(SWEEPS_PER_STEP)
    sampler = ClockSampler(local)
    launches0 = lib.pi_launch_count(eng._engine)
    barrier()
    if rank == 0:
        sampler.start()
    t0 = time.perf_counter()
    dev_ms = 0.0
    for _ in range(args.steps):
        residual, ms = eng.sweeps(SWEEPS_PER_STEP)
        dev_ms += ms
    barrier()
    wall_s = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    launches = lib.pi_launch_count(eng._engine) - launches0
    if td is not None:
        t = torch.tensor([dev_ms], device="cuda", dtype=torch.float64)
        td.all_reduce(t, op=td.ReduceOp.MAX)
        dev_ms = float(t.item())
    ms_per_step = dev_ms / args.steps
    value = N * SWEEPS_PER_STEP / (ms_per_step * 1e-3)
    # checksum of V after 2 x 25 + (warmup + steps) x 25 sweeps: the same point of the same protocol in the reference arm
    v_local = torch.as_tensor(eng.d_value_function, device=f"cuda:{local}")[lo:hi]
    csum = torch.tensor([v_checksum(v_local)], device="cuda", dtype=torch.int64)
    if td is not None:
        td.all_reduce(csum, op=td.ReduceOp.SUM)
    csum = int(csum.item())
    n_sweeps_at_checksum = 2 * SWEEPS_PER_STEP + (max(args.warmup, 3) + args.steps) * SWEEPS_PER_STEP
    kinfo = eng.eval_kernel_info()   # which sweep kernel the engine runs for THIS policy (scalar gather / x-line)
    if args.dump_outputs:
        values, _ = eng.download()   # every rank: the whole V is gathered when sharded
        if rank == 0:
            dump_outputs(args.dump_outputs, values, residual)
        del values

    # ---- end-to-end arm: host buffers in, host buffers out ---------------------
    n_local = hi - lo
    pol_host = torch.empty(n_local, dtype=torch.int32).pin_memory()
    v_host = torch.empty(n_local, dtype=torch.float32).pin_memory()
    pol_np, v_np = pol_host.numpy(), v_host.numpy()
    _ffi.check(lib.pi_copy_local_results(eng._engine, None, _ffi.ptr(pol_np)))      # this rank's slice, storage order

    def e2e_step():
        _ffi.check(lib.pi_upload_policy_local(eng._engine, _ffi.ptr(pol_np)))     # H2D policy slice + row compaction
        d, _ = eng.sweeps(SWEEPS_PER_STEP)
        _ffi.check(lib.pi_copy_local_results(eng._engine, _ffi.ptr(v_np), None))  # D2H value slice
        return d

    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    if td is not None:
        t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
        td.all_reduce(t, op=td.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = N * SWEEPS_PER_STEP * args.steps / e2e_s

    out = None
    if rank == 0:
        D = eng.N_DIMS
        bytes_per_backup = (D + 2) * 4 + 4 + 4          # compact row + V read + V write
        peak, peak_src = measured_peak()
        per_gpu_backups = value / world
        achieved = per_gpu_backups * bytes_per_backup / 1e9
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.bins, eng.n_actions, eng.config.gamma,
                                      ("contiguous state ranges, needs-driven V exchange: " + os.environ.get("DPB200_EXCHANGE", "p2p") +
                                       " (p2p = peer stores fused into the sweep kernel over CUDA IPC / NVLink + barrier kernel; nccl = grouped send/recv)")
                                      if world > 1 else "single GPU"),
            "v_checksum": csum, "v_checksum_after_sweeps": n_sweeps_at_checksum,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(n_local * 4),
                    "d2h_bytes_per_step": int(n_local * 4 + 4),
                    "call": "pi_upload_policy_local + pi_sweeps(25) + pi_copy_local_results (pinned host buffers, each rank its own slice)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic(args.bins), "kernel": kinfo["kernel"],
                         "peak_source": peak_src, "layout": "compact row (base + D fractions + reward)",
                         "algorithmic_bytes_per_backup": bytes_per_backup,
                         "survey_gather_counted_bytes_per_backup": (D + 2) * 4 + 4 * (1 << D) + 13,
                         "per_gpu": world > 1},
            "table_build": {"ms": build_ms, "rows_per_s": (hi - lo) * eng.n_actions / (build_ms * 1e-3),
                            "bytes": int(lib.pi_table_bytes(eng._engine))},
            "wall_s_timed_region": wall_s,
        }
        W = D + 2
        out["stages"] = {"K5": {
            "config": f"{ENV} --bins {args.bins}",
            "build": stage(build_ms, (hi - lo) * eng.n_actions, W * 4, "rows"),
            "eval": stage(ms_per_step / SWEEPS_PER_STEP, hi - lo, W * 4 + 8, "backups"),
            "improve": stage(improve_ms, hi - lo, eng.n_actions * W * 4 + W * 4 + 8, "states"),
            "per_gpu": world > 1}}
    eng.close()
    # K5 run to a stable policy through the public API (every rank takes part when sharded)
    if not args.no_stable:
        st = run_to_stable(ENV, args.bins, local, pdist.make_shard(local) if world > 1 else None)
        if rank == 0:
            out["k5_to_stable"] = st
    if rank == 0:
        if not args.no_extras and world == 1:
            out["stages"].update(small_config_stages())
            out["k5_bins12_to_stable"] = run_to_stable(ENV, 12, local, None)
        # K1 first: the OpenMP workers of the CPU baseline keep spinning for a while after their last
        # parallel region and would be charged to the small-grid run (host-side latency matters there)
        if not args.no_converge and world == 1:
            out["time_to_converge"] = time_to_converge()
        if not args.no_cpu_baseline and world == 1:
            out["cpu_baseline"] = cpu_baseline(args.bins)
    if td is not None:
        td.barrier()
        td.destroy_process_group()
    return out


def stage(ms: float, units: int, bytes_per_unit: int, unit: str) -> dict:
    """One stage of one configuration: device time, throughput, algorithmic HBM bytes and roofline fraction."""
    peak, _ = measured_peak()
    gbs = units * bytes_per_unit / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
    return {"ms": ms, f"{unit}_per_s": units / (ms * 1e-3) if ms > 0 else 0.0, "algorithmic_bytes_per_unit": bytes_per_unit,
            "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peak}


# BASELINE.json configs[0..3]; K2 also with the fine action grid its description names (201 actions)
SMALL_CONFIGS = [
    ("K1", "pendulum", 200, None),
    ("K2", "continuous_mountain_car", 400, None),
    ("K2-fine", "continuous_mountain_car", 400, 201),
    ("K3", "cartpole", 30, None),
    ("K4", "double_pendulum_swingup", 50, None),
]


def small_config_stages() -> dict:
    """Per configuration K1-K4 and per stage (table build / evaluation sweep / improvement pass): device ms, throughput,
    algorithmic bytes, fraction of the HBM roofline — and the reference's own kernels for the same stage beside it
    (oracle/_ref cubins; eval = its evaluation kernel + max|x-y| reduction per sweep)."""
    import torch

    from dynamicprogramming_b200 import envs
    from oracle import ref_runner

    out = {}
    for tag, env, bins, n_act in SMALL_CONFIGS:
        spec = envs.REGISTRY[env]
        actions = None
        if n_act is not None:
            actions = np.linspace(float(spec.actions.min()), float(spec.actions.max()), n_act).astype(np.float32)
        eng = spec.make(bins=bins, actions=actions)
        eng.build_table()
        eng.sweeps(2 * SWEEPS_PER_STEP)
        eng.policy_improvement()                       # a mixed policy, as in the K5 protocol
        st0 = eng.engine_stats()
        eng.sweeps(8 * SWEEPS_PER_STEP)               # warm
        _, ms = eng.sweeps(40 * SWEEPS_PER_STEP)
        eng.policy_improvement()
        st1 = eng.engine_stats()
        N, A, W = eng.n_states, eng.n_actions, eng.N_DIMS + 2
        rec = {"config": f"{env} --bins {bins}, {A} actions, {N:,} states", "kernel": eng.eval_kernel_info()["kernel"],
               "build": stage(st1["build_ms"], N * A, W * 4, "rows"),
               "eval": stage(ms / (40 * SWEEPS_PER_STEP), N, W * 4 + 8, "backups"),
               "improve": stage(st1["improve_ms"] - st0["improve_ms"], N, A * W * 4 + W * 4 + 8, "states")}
        eng.close()
        if ref_runner.available(env):
            ref = ref_runner.from_engine_env(env, bins=bins, actions=actions)
            for _ in range(2 * SWEEPS_PER_STEP):
                ref.eval_launch()
                ref.d_value_function, ref.d_new_value_function = ref.d_new_value_function, ref.d_value_function
            ref.improve_launch()
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            n = 4 * SWEEPS_PER_STEP
            torch.cuda.synchronize()
            e0.record()
            for _ in range(n):
                ref.eval_launch()
                ref._max_abs_diff()
                ref.d_value_function, ref.d_new_value_function = ref.d_new_value_function, ref.d_value_function
            e1.record()
            ref.improve_launch()
            e2.record()
            torch.cuda.synchronize()
            rec["reference_kernels"] = {"eval_ms_per_sweep": e0.elapsed_time(e1) / n, "improve_ms": e1.elapsed_time(e2)}
            del ref
            torch.cuda.empty_cache()
        out[tag] = rec
    return out


def run_to_stable(env: str, bins: int, device: int, shard) -> dict:
    """run() to a stable policy through the public API: table build, every evaluation and improvement, D2H."""
    from dynamicprogramming_b200 import envs

    spec = envs.REGISTRY[env]
    t0 = time.perf_counter()
    eng = spec.make(bins=bins, device=device, shard=shard)
    t1 = time.perf_counter()
    eng.run()
    t2 = time.perf_counter()
    return {"workload": f"{env} --bins {bins} ({eng.n_states:,} states x {eng.n_actions} actions), run() to a stable policy "
                        "incl. table build and D2H", "seconds": t2 - t1, "create_seconds": t1 - t0,
            "pi_iterations": eng.pi_iterations, "eval_sweeps": eng.total_eval_sweeps, "converged": bool(eng.converged),
            "eval_ms": eng.stats["eval_ms"], "improve_ms": eng.stats["improve_ms"], "build_ms": eng.stats["build_ms"]}


def cpu_baseline(bins: int, budget_s: float = 12.0) -> dict:
    """CPU restatement (oracle port) on the first two dim-0 slabs of the same grid."""
    from dynamicprogramming_b200 import envs
    from oracle import cpu_oracle

    spec = envs.REGISTRY[ENV]
    axes = [np.asarray(v, np.float32) for v in spec.bins_space(bins).values()]
    slabs = 2
    sub = [axes[0][:slabs]] + axes[1:]
    cfg = spec.config()
    o = cpu_oracle.CpuPolicyIteration(ENV, sub, spec.actions, cfg.gamma, cfg.theta, 10, 1)
    D = len(axes)
    st = 1
    for d in range(D - 1, -1, -1):
        o.grid.shape[d] = bins
        o.grid.strides[d] = st
        o.grid.lo[d] = float(axes[d][0])
        o.grid.hi[d] = float(axes[d][-1])
        st *= bins
    V = np.zeros(bins ** D, np.float32)
    o.policy[:] = np.random.default_rng(0).integers(0, len(spec.actions), o.n_states).astype(np.int32)
    o.eval_sweep(V)  # warm-up
    t0 = time.perf_counter()
    n = 0
    while True:
        o.eval_sweep(V)
        n += 1
        if time.perf_counter() - t0 > budget_s or n >= 8:
            break
    dt = time.perf_counter() - t0
    return {"value": o.n_states * n / dt, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
            "sample": f"{n} sweeps over the first {slabs} of {bins} dim-0 slabs ({o.n_states:,} of {bins ** D:,} states), "
                      f"oracle/pi_oracle.c with OpenMP on all host cores"}


def time_to_converge() -> dict:
    """Config K1 (Pendulum --bins 200) run to the end through the public API."""
    from dynamicprogramming_b200 import envs

    eng = envs.make("pendulum")
    t0 = time.perf_counter()
    eng.run()
    dt = time.perf_counter() - t0
    return {"workload": "pendulum 2-D --bins 200 (40,000 states x 21 actions), run() incl. table build and D2H",
            "seconds": dt, "pi_iterations": eng.pi_iterations, "eval_sweeps": eng.total_eval_sweeps,
            "converged": bool(eng.converged),
            "note": "the policy keeps changing until max_pi_iter = 50 in both arms (same counts as the reference loop)",
            "eval_ms": eng.stats["eval_ms"], "improve_ms": eng.stats["improve_ms"]}


# ---------------------------------------------------------------------- reference
def run_reference(args) -> dict | None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    import torch

    from dynamicprogramming_b200 import envs
    from oracle import ref_runner

    spec = envs.REGISTRY[ENV]
    N = args.bins ** 6
    cfg_desc = workload_config(args.bins, len(spec.actions), spec.config().gamma, "single GPU")
    csum = None
    if ref_runner.available(ENV) and torch.cuda.is_available():
        torch.cuda.set_device(0)
        ref = ref_runner.from_engine_env(ENV, bins=args.bins)
        # same policy protocol as our arm: bounded evaluation, one improvement
        for _ in range(2 * SWEEPS_PER_STEP):
            ref.eval_launch()
            ref.d_value_function, ref.d_new_value_function = ref.d_new_value_function, ref.d_value_function
        ref.improve_launch()

        def step():
            # policy_evaluation inner loop (:305-326): eval kernel + max|x-y| each sweep, one .get() per 25
            for i in range(SWEEPS_PER_STEP):
                ref.eval_launch()
                d = ref._max_abs_diff()
                ref.d_value_function, ref.d_new_value_function = ref.d_new_value_function, ref.d_value_function
            return float(d.item())

        for _ in range(max(args.warmup, 3)):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms_per_step = e0.elapsed_time(e1) / args.steps
        value = N * SWEEPS_PER_STEP / (ms_per_step * 1e-3)
        csum = v_checksum(ref.d_value_function)
        e2 = torch.cuda.Event(enable_timing=True)
        e1.record()
        ref.improve_launch()
        e2.record()
        torch.cuda.synchronize()
        ref_stages = {"K5": {"eval_ms_per_sweep": ms_per_step / SWEEPS_PER_STEP, "improve_ms": e1.elapsed_time(e2)}}
        del ref
        torch.cuda.empty_cache()
        # K1 (pendulum --bins 200) to the end with the reference's kernels and host loop, like our arm's
        # time_to_converge: run() only (kernels are already compiled on both sides), D2H included
        ttc = None
        if not args.no_converge:
            ref1 = ref_runner.from_engine_env("pendulum")
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ref1.run()
            ttc = {"workload": "pendulum 2-D --bins 200 (40,000 states x 21 actions), reference kernels + reference host loop, run() incl. D2H",
                   "seconds": time.perf_counter() - t0, "pi_iterations": ref1.pi_iterations, "eval_sweeps": ref1.total_sweeps,
                   "converged": bool(ref1.converged)}
        k5_12 = None
        if not args.no_extras:
            # the autoresearch trial workload (runners/trial_runner.sh: --bins 12) to a stable policy with the reference's
            # kernels and host loop
            ref12 = ref_runner.from_engine_env(ENV, bins=12)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ref12.run()
            k5_12 = {"workload": f"{ENV} --bins 12 ({ref12.n_states:,} states), reference kernels + reference host loop, run() incl. D2H",
                     "seconds": time.perf_counter() - t0, "pi_iterations": ref12.pi_iterations, "eval_sweeps": ref12.total_sweeps,
                     "converged": bool(ref12.converged)}
        kind = {"value": value, "unit": UNIT, "cores": 0, "kind": "reference",
                "sample": "the reference's own eval kernel + max|x-y| reduction (oracle/_ref cubin, NVRTC-compiled "
                          "from the original project's sources) on one B200, full grid; the reference has no CPU path"}
    else:
        cb = cpu_baseline(args.bins, budget_s=30.0)
        value = cb["value"]
        ms_per_step = N * SWEEPS_PER_STEP / value * 1e3
        kind = dict(cb)
        ttc = None
        k5_12 = None
        ref_stages = None
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg_desc, "cpu_baseline": kind,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if csum is not None:
        out["v_checksum"] = csum
        out["v_checksum_after_sweeps"] = 2 * SWEEPS_PER_STEP + (max(args.warmup, 3) + args.steps) * SWEEPS_PER_STEP
    if ttc is not None:
        out["time_to_converge"] = ttc
    if k5_12 is not None:
        out["k5_bins12_to_stable"] = k5_12
    if ref_stages is not None:
        out["stages"] = ref_stages
    return out


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--bins", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-converge", action="store_true")
    ap.add_argument("--no-stable", action="store_true", help="skip the K5 run to a stable policy")
    ap.add_argument("--no-extras", action="store_true", help="skip the per-configuration stage table (K1-K4) and the --bins 12 runs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write V and the residual after the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs is only available with --impl ours")
    _quiet_logs()
    # stdout carries exactly ONE JSON line: while the benchmark runs, file descriptor 1 points at stderr, so
    # anything a library prints there (torch's "NCCL version ..." banner under torchrun) cannot precede it
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        out = run_reference(args) if args.impl == "reference" else run_ours(args)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    if out is not None:
        print(json.dumps(out), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
