#!/usr/bin/env python3
"""K5 (double cartpole swing-up 6-D, --bins 20) under the bench policy: the plane-staged sweep in several
configurations vs the gather sweep (CUDA-event timings, bitwise comparison, plan statistics).
    python scripts/exp_plane.py [bins] [cfg ...]"""
import json, os, sys, time
from pathlib import Path
ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
os.environ.setdefault("DPB200_PLANE", "off")
from dynamicprogramming_b200 import envs
try:
    from loguru import logger
    logger.remove(); logger.add(sys.stderr, level="INFO")
except ImportError:
    pass
bins = int(sys.argv[1]) if len(sys.argv) > 1 else 20
cfgs = sys.argv[2:] or ["0,0,2,2,2", "0,0,2,2,0", "0,0,2,1,2", "0,0,2,3,2", "0,10,2,2,2", "0,0,3,2,2"]
t0 = time.time()
eng = envs.make("double_cartpole_swingup", bins=bins)
eng.build_table()
print("layout", eng.layout(), "kernel", eng.eval_kernel_info(), flush=True)
eng.sweeps(50)
eng.policy_improvement()
print("setup %.1f s; kernel for the bench policy: %s" % (time.time() - t0, eng.eval_kernel_info()["kernel"]), flush=True)
d, ms = eng.sweeps(25)
print("engine sweeps: %.4f ms/sweep" % (ms / 25), flush=True)
out = []
for cfg in cfgs:
    # "cfg@K=V;K=V": environment variables set while this configuration is compiled and timed
    spec, _, envs_ = cfg.partition("@")
    for kv in filter(None, envs_.split(";")):
        k, _, v = kv.partition("=")
        os.environ[k] = v
    try:
        r = eng.debug_plane(spec, iters=10)
    except Exception as ex:  # noqa: BLE001
        r = {"error": str(ex)[:300]}
    r["cfg"] = cfg
    for kv in filter(None, envs_.split(";")):
        os.environ.pop(kv.partition("=")[0], None)
    print(json.dumps(r), flush=True)
    out.append(r)
(ROOT / "gpurun_out").mkdir(exist_ok=True)
(ROOT / "gpurun_out" / f"exp_plane_{bins}.json").write_text(json.dumps(out, indent=1))
