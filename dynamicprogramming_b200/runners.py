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
mean return, mean discounted return, mean length, fraction of episodes that terminated.
"""
from __future__ import annotations

import argparse
import sys
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
    p.add_argument("--bins", type=int, default=spec.default_bins, help=f"Bins per dimension (default: {spec.default_bins})")
    p.add_argument("--seed", type=int, default=42, help="Random seed of the queried states (default: 42)")
    p.add_argument("--no-plot", action="store_true", help="Accepted for compatibility (plots are never produced)")
    p.add_argument("--retrain", action="store_true", help="Force retraining even if a saved policy exists")
    p.add_argument("--save-path", type=Path, default=Path(f"results/{runner}_policy.npz"))
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


def rollout_summary(pi, episodes: int, steps: int, seed: int, gamma: float) -> dict:
    """--rollout: closed-loop episodes from start_states() under the plugin's dynamics (pi.rollout)."""
    res = pi.rollout(start_states(pi, episodes, seed), steps, gamma=gamma)
    return {"episodes": episodes, "steps": steps, "mean_return": float(res.total_reward.mean()),
            "mean_discounted_return": float(res.discounted_return.mean()), "mean_length": float(res.length.mean()),
            "terminated": float(res.terminated.mean())}


def format_rollout(r: dict) -> str:
    return (f"[=] rollout {r['episodes']} episodes x {r['steps']} steps | mean return {r['mean_return']:.6f} | "
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
        pi = train(runner, args.save_path, bins=args.bins, **kw)
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
        print(format_rollout(rollout_summary(pi, args.episodes, args.steps, args.seed, gamma)))
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
