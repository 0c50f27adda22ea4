"""The built-in environment specs (dynamicprogramming_b200.envs.REGISTRY — what tests, bench.py and the reference arm
build their grids and action sets from) must equal what the reference's runners declare (BINS_SPACE, ACTION_SPACE of
runners/*_cuda.py).  tests/golden/reference_manifest.json stores them in the layout of the "envs" part of the manifest
oracle/build_ref.py writes from those runners (its "source" entry says where the values come from), so the check runs
without the original project."""
import json
from pathlib import Path

import numpy as np

from dynamicprogramming_b200 import envs

MANIFEST = Path(__file__).resolve().parent / "golden" / "reference_manifest.json"


def test_registry_equals_the_reference_manifest():
    man = json.loads(MANIFEST.read_text())["envs"]
    assert set(man) == set(envs.REGISTRY)
    for name, meta in man.items():
        spec = envs.REGISTRY[name]
        assert spec.cls.N_DIMS == meta["D"], name
        space = spec.bins_space(None)
        assert list(space) == list(meta["bins"]), name           # same axis names, same order
        for key, (lo, hi, n) in meta["bins"].items():
            ax = np.asarray(space[key], dtype=np.float32)
            assert len(ax) == n, (name, key)
            assert np.float32(ax[0]) == np.float32(lo) and np.float32(ax[-1]) == np.float32(hi), (name, key)
        np.testing.assert_array_equal(np.asarray(spec.actions, np.float32), np.asarray(meta["actions"], np.float32))
