"""
Command line of the reference's runners (runners/*_cuda.py `__main__` blocks, e.g.
runners/pendulum_cuda.py:264-309; README.md "CLI Reference" :327-345) on top of the B200 engine:

    python -m dynamicprogramming_b200.runners pendulum_cuda --bins 200 --retrain
    python -m dynamicprogramming_b200.runners double_cartpole_swingup_cuda --bins 12 --no-plot

Same runner names, same flags, same train-or-load behaviour (`--save-path` exists and no
`--retrain` => `Cls.load`, no GPU touched; otherwise `train()` = construct, `run()`, `save()`),
same `--bins` semantics (endpoints re-read from the default float32 grid), same saved-policy
`.npz`.  What the reference does AFTER training — gymnasium / pygame roll-outs, videos and
matplotlib plots (`evaluate`, `evaluate_random`, `plot_*`) — is outside the hot path (SURVEY §2
rows 5-7; those packages are not in this image): `--render`, `--record`, `--random` and the plots
are accepted and reported as skipped.  Instead the runner prints a summary of the solution and, as
a smoke check of the inference path, queries `--episodes` random states through the batched
`get_optimal_action` (include/dpb200.h: pi_lookup_*).

With `--rollout` it also runs what evaluate() runs — the policy in closed loop — on the device:
`--episodes` episodes of up to `--steps` steps from the same seeded uniform start states, simulated
with the plugin's own float32 `step_dynamics` (the model the DP solved, not gymnasium;
include/dpb200.h: pi_rollout_*), discounted with the runner's gamma, and prints one summary line:
mean return, mean discounted return, mean length, fraction of episodes that terminated.  `--rollout-controller
lookahead` acts with the one-step lookahead on the value function instead of the interpolated grid policy
(engine.lookahead); the summary line then names the controller.

With `--warm-start-bins B` a training run first solves the same runner with the same config at `B` bins and starts
the `--bins` solve from that value function (engine.warm_start); `--warm-start-from PATH` starts it from a saved
policy's value function instead.  Either flag adds one line per solve: bins, PI iterations, evaluation sweeps and
host seconds (construction, warm start and run(), not the save).
"""
from __future__ import annotations

import argparse
import sys
import time
from pathlib import Path

import numpy as np

from . import envs

# reference runner file name -> built-in environment
RUNNERS = {
    "pendulum_cuda": "pendulum",
    "mountain_car_cuda": "mountain_car",
    "continuous_mountain_car_cuda": "continuous_mountain_car",
    "cartpole_cuda": "cartpole",
    "cartpole_swingup_cuda": "cartpole_swingup",
    "double_pendulum_swingup_cuda": "double_pendulum_swingup",
    "overhead_crane_cuda": "overhead_crane",
    "double_cartpole_cuda": "double_cartpole",
    "double_cartpole_swingup_cuda": "double_cartpole_swingup",
}


def build_parser(runner: str) -> argparse.ArgumentParser:
    spec = envs.REGISTRY[RUNNERS[runner]]
    p = argparse.ArgumentParser(prog=f"python -m dynamicprogramming_b200.runners {runner}",
                                description=f"{runner} — CUDA Policy Iteration (B200 engine)")
    p.add_argument("--render", action="store_true", help="(skipped: pygame roll-outs are outside the DP path)")
    p.add_argument("--random", type=int, nargs="?", const=5, default=None, metavar="N",
                   help="(skipped: random-policy gymnasium episodes)")
    p.add_argument("--record", type=Path, default=None, metavar="PATH", help="(skipped: video recording)")
    p.add_argument("--episodes", type=int, default=5,
                   help="Number of states queried through get_optimal_action (and of episodes with --rollout)")
    p.add_argument("--steps", type=int, default=1000, help="Steps per episode with --rollout (else accepted for compatibility)")
    p.add_argument("--rollout", action="store_true",
                   help="Also run --episodes closed-loop episodes of --steps steps on the GPU with the plugin's dynamics")
    p.add_argument("--rollout-controller", choices=("policy", "lookahead"), default="policy",
                   help="What acts in --rollout episodes: the interpolated grid policy (default) or the one-step "
                        "lookahead on the value function")
    p.add_argument("--bins", type=int, default=spec.default_bins, help=f"Bins per dimension (default: {spec.default_bins})")
    p.add_argument("--seed", type=int, default=42, help="Random seed of the queried states (default: 42)")
    p.add_argument("--no-plot", action="store_true", help="Accepted for compatibility (plots are never produced)")
    p.add_argument("--retrain", action="store_true", help="Force retraining even if a saved policy exists")
    p.add_argument("--save-path", type=Path, default=Path(f"results/{runner}_policy.npz"))
    warm = p.add_mutually_exclusive_group()
    warm.add_argument("--warm-start-bins", type=int, default=None, metavar="B",
                      help="When training: first solve at B bins, then start the --bins solve from its value function")
    warm.add_argument("--warm-start-from", type=Path, default=None, metavar="PATH",
                      help="When training: start the --bins solve from the value function of a saved policy (.npz)")
    if runner == "overhead_crane_cuda":
        p.add_argument("--start-x", type=float, default=2.5, help="Accepted for compatibility (roll-out start)")
        p.add_argument("--target-x", type=float, default=-2.5, help="Target trolley position (m), baked into the CUDA source")
    return p


def train(runner: str, save_path: Path, bins: int | None = None, **kw):
    """The reference's train(): construct with the runner's config, run(), save()
    (e.g. runners/pendulum_cuda.py:116-130)."""
    spec = envs.REGISTRY[RUNNERS[runner]]
    pi = spec.make(bins=bins, **kw)
    pi.run()
    pi.save(save_path)
    return pi


def train_warm(runner: str, save_path: Path, bins: int | None = None, warm_bins: int | None = None,
               warm_from: Path | None = None, **kw):
    """train() started from a coarser solution: a solve at `warm_bins` (same runner, same config), or the saved policy
    `warm_from`, warm-starts the solve at `bins` (engine.warm_start).  Returns the trained engine and one dict per solve
    (bins, PI iterations, evaluation sweeps, host seconds)."""
    spec = envs.REGISTRY[RUNNERS[runner]]
    solves = []

    def solve(b, source=None):
        t0 = time.perf_counter()
        pi = spec.make(bins=b, **kw)
        if source is not None:
            pi.warm_start(source)
        pi.run()
        solves.append({"bins": spec.default_bins if b is None else int(b), "pi_iterations": pi.pi_iterations, "sweeps": pi.total_eval_sweeps,
                       "seconds": time.perf_counter() - t0})
        return pi

    source = solve(warm_bins) if warm_from is None else warm_from
    pi = solve(bins, source)
    pi.save(save_path)
    return pi, solves


def format_solve(s: dict) -> str:
    return (f"[=] solve at {s['bins']} bins | {s['pi_iterations']} PI iterations | {s['sweeps']} evaluation sweeps | "
            f"{s['seconds']:.2f} s")


def start_states(pi, n: int, seed: int) -> np.ndarray:
    """`n` seeded uniform states inside the grid's bounds: the states summarize() queries and --rollout starts from."""
    rng = np.random.default_rng(seed)
    return (pi.bounds_low + (pi.bounds_high - pi.bounds_low) * rng.random((n, len(pi.bounds_low)))).astype(np.float32)


def summarize(pi, n_queries: int, seed: int) -> dict:
    hist = np.bincount(pi.policy, minlength=len(pi.action_space))
    out = {"states": int(pi.policy.size), "V_min": float(pi.value_function.min()), "V_max": float(pi.value_function.max()),
           "policy_histogram": hist.tolist()}
    if n_queries > 0:
        pts = start_states(pi, n_queries, seed)
        out["queried_states"] = pts.tolist()
        out["interpolated_actions"] = pi.lookup_actions(pts).tolist()
    return out


def rollout_summary(pi, episodes: int, steps: int, seed: int, gamma: float, controller: str = "policy") -> dict:
    """--rollout: closed-loop episodes from start_states() under the plugin's dynamics (pi.rollout)."""
    res = pi.rollout(start_states(pi, episodes, seed), steps, gamma=gamma, controller=controller)
    out = {"episodes": episodes, "steps": steps, "mean_return": float(res.total_reward.mean()),
           "mean_discounted_return": float(res.discounted_return.mean()), "mean_length": float(res.length.mean()),
           "terminated": float(res.terminated.mean())}
    if controller != "policy":
        out["controller"] = controller
    return out


def format_rollout(r: dict) -> str:
    who = f" ({r['controller']} controller)" if "controller" in r else ""
    return (f"[=] rollout{who} {r['episodes']} episodes x {r['steps']} steps | mean return {r['mean_return']:.6f} | "
            f"mean discounted return {r['mean_discounted_return']:.6f} | mean length {r['mean_length']:.2f} | "
            f"terminated {r['terminated']:.4f}")


def main(argv: list[str] | None = None) -> int:
    argv = list(sys.argv[1:] if argv is None else argv)
    if not argv or argv[0] in ("-h", "--help") or argv[0] not in RUNNERS:
        print("usage: python -m dynamicprogramming_b200.runners <runner> [options]\nrunners: " + ", ".join(RUNNERS))
        return 0 if argv and argv[0] in ("-h", "--help") else 2
    runner = argv[0]
    args = build_parser(runner).parse_args(argv[1:])
    spec = envs.REGISTRY[RUNNERS[runner]]
    if args.random is not None:
        print("[!] --random: random-policy gymnasium episodes are outside the DP path; nothing to do")
        return 0
    kw = {}
    if runner == "overhead_crane_cuda":
        kw["target_x"] = float(args.target_x)
    if args.save_path.exists() and not args.retrain:
        print(f"[+] Loading existing policy from {args.save_path}")
        pi = spec.cls.load(args.save_path)
    else:
        print("[*] Training new policy...")
        if args.warm_start_bins is None and args.warm_start_from is None:
            pi = train(runner, args.save_path, bins=args.bins, **kw)
        else:
            pi, solves = train_warm(runner, args.save_path, bins=args.bins, warm_bins=args.warm_start_bins,
                                    warm_from=args.warm_start_from, **kw)
            for s_ in solves:
                print(format_solve(s_))
    for flag, what in ((args.render, "--render"), (args.record, "--record")):
        if flag:
            print(f"[!] {what}: rendering / recording needs gymnasium + pygame and is outside the DP path; skipped")
    s = summarize(pi, args.episodes, args.seed)
    print(f"[=] {s['states']:,} states | V in [{s['V_min']:.4f}, {s['V_max']:.4f}] | policy histogram {s['policy_histogram']}")
    for p_, a_ in zip(s.get("queried_states", []), s.get("interpolated_actions", [])):
        print("    state " + np.array2string(np.asarray(p_), precision=3) + f" -> action {a_:.4f}")
    if args.rollout and args.episodes > 0:
        # the runner's gamma: a loaded policy carries the default CudaPIConfig, not the one it was trained with
        gamma = float(np.float32(spec.config().gamma))
        print(format_rollout(rollout_summary(pi, args.episodes, args.steps, args.seed, gamma, args.rollout_controller)))
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
