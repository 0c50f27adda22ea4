#!/usr/bin/env python3
"""Time tuning variants of the scalar evaluation sweep at K5 under a REAL converged policy
(scripts/data/k5_policy16.npz, captured by scripts/k5_policies.py; falls back to the bench policy).
Every variant must produce the same V bits.

    python scripts/exp_variants.py "DPB200_EVAL_VARIANT=0" "DPB200_EVAL_VARIANT=1" "DPB200_EVAL_VARIANT=64" ...
"""
import hashlib, os, sys, time
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
os.environ.setdefault("DPB200_XLINE", "off")
from loguru import logger
logger.remove()
import numpy as np
from dynamicprogramming_b200 import envs

cfgs = sys.argv[1:] or ["DPB200_EVAL_VARIANT=0"]
ENV, BINS = os.environ.get("EXP_ENV", "double_cartpole_swingup"), int(os.environ.get("EXP_BINS", "20"))
pol_file = Path(__file__).resolve().parent / "data" / "k5_policy16.npz"
policy = np.load(pol_file)["policy"].astype(np.int32) if pol_file.exists() and (ENV, BINS) == ("double_cartpole_swingup", 20) else None
print(f"== {ENV} --bins {BINS}, policy: {'converged (captured)' if policy is not None else 'greedy after 50 sweeps of policy 0'}", flush=True)
ref_hash = None
for cfg in cfgs:
    kv = dict(x.split("=", 1) for x in cfg.split())
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update(kv)
    eng = envs.make(ENV, bins=BINS)
    eng.build_table()
    if policy is not None:
        eng.upload_policy(policy)
    else:
        eng.sweeps(50); eng.policy_improvement()
        eng.upload_values(np.zeros(eng.n_states, np.float32))
    n_sw = 25 if eng.n_states > 4_000_000 else 200
    eng.sweeps(n_sw)
    ms = []
    for _ in range(4):
        ms.append(eng.sweeps(n_sw)[1] / n_sw)
    v, _ = eng.download()
    h = hashlib.sha1(v.tobytes()).hexdigest()[:12]
    ref_hash = ref_hash or h
    print(f"{cfg:60s} ms/sweep min {min(ms):.4f} med {sorted(ms)[len(ms)//2]:.4f}  V {h} {'OK' if h == ref_hash else 'MISMATCH'}  [{eng.eval_kernel_info()["kernel"][:58]}]", flush=True)
    eng.close()
    for k, v0 in old.items():
        if v0 is None: os.environ.pop(k, None)
        else: os.environ[k] = v0
