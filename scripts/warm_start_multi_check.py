#!/usr/bin/env python3
"""torchrun --nproc-per-node N scripts/warm_start_multi_check.py — a sharded warm start + run() equals the single-GPU
one, bit for bit (tests/test_gpu_warm_start.py).

Every rank solves the coarse grid unsharded, warm-starts its shard of the fine grid from it (pi_prolong_values is
collective: each rank prolongs its slice, the full V is all-gathered) and runs; rank 0 also does the same on one GPU
and compares V, policy, PI iterations and sweep counts."""
import json
import os
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from loguru import logger

logger.remove()
import torch

from dynamicprogramming_b200 import dist as pdist, envs

rank = int(os.environ.get("RANK", 0))
local = int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
td = pdist.init_process_group()
# (env, coarse bins, fine bins, max_pi_iter, engine environment of the sharded run)
cases = [("cartpole", 7, 12, 4, {}), ("double_cartpole_swingup", 5, 8, 2, {}),
         ("double_cartpole_swingup", 5, 8, 2, {"DPB200_PLANE": "force"}), ("pendulum", 17, 33, 6, {})]
ok = True
for env, coarse_bins, bins, max_pi, engine_env in cases:
    for k in ("DPB200_FAST_DIM", "DPB200_XLINE", "DPB200_PAIR", "DPB200_PLANE", "DPB200_EXCHANGE"):
        os.environ.pop(k, None)
    spec = envs.REGISTRY[env]
    cfg = spec.config()
    cfg.max_pi_iter = max_pi
    coarse = spec.make(bins=coarse_bins, config=cfg, device=local)
    coarse.run()
    os.environ.update(engine_env)
    eng = spec.make(bins=bins, config=cfg, device=local, shard=pdist.make_shard(local))
    ws = eng.warm_start(coarse)
    eng.run()
    res = dict(env=env, bins=bins, coarse_bins=coarse_bins, pi=eng.pi_iterations, sweeps=eng.total_eval_sweeps,
               changed=ws["changed"], sharded_env=engine_env)
    if rank == 0:
        for k in engine_env:
            os.environ.pop(k, None)
        one = spec.make(bins=bins, config=cfg, device=local)
        ws1 = one.warm_start(coarse)
        one.run()
        res.update(pi_1gpu=one.pi_iterations, sweeps_1gpu=one.total_eval_sweeps, changed_1gpu=ws1["changed"],
                   policy_diff=int(np.sum(one.policy != eng.policy)),
                   v_bitdiff=int(np.sum(one.value_function.view(np.uint32) != eng.value_function.view(np.uint32))))
        good = (res["policy_diff"] == 0 and res["v_bitdiff"] == 0 and res["pi"] == res["pi_1gpu"]
                and res["sweeps"] == res["sweeps_1gpu"] and res["changed"] == res["changed_1gpu"])
        ok &= good
        print(("OK   " if good else "FAIL ") + json.dumps(res), flush=True)
    td.barrier()
flag = torch.tensor([1 if ok else 0], device="cuda")
td.broadcast(flag, src=0)
td.destroy_process_group()
sys.exit(0 if int(flag.item()) else 1)
