import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

os.environ.setdefault("LOGURU_LEVEL", "WARNING")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    try:
        from loguru import logger

        logger.remove()
        logger.add(sys.stderr, level="WARNING")
    except ImportError:
        pass


def _has_cuda() -> bool:
    try:
        from dynamicprogramming_b200 import _ffi

        return _ffi.lib().pi_device_count() > 0
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_cuda():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden_dir() -> Path:
    return ROOT / "tests" / "golden"


REFERENCE_GOLDEN = ROOT / "tests" / "golden" / "reference_parity.json"


class ReferenceGolden:
    """What the reference's own kernels computed for one test case, stored in tests/golden/reference_parity.json
    (its "source" entry says how it was produced): per array its dtype, shape, the SHA-256 of its bytes and the values
    at a few flat positions (`at`, `sample`) for the failure message; scalars as they are.  `check` is bit-exact, as
    a comparison with the reference's arrays themselves would be.

    The file is data, not output of this suite: nothing here writes it.  A new or changed case must be recorded from
    the reference's kernels (oracle/_ref, oracle/ref_runner.py), never from the engine under test."""

    def __init__(self, case: str, stored: dict | None) -> None:
        self.case, self.stored = case, stored

    def _expected(self, label: str):
        assert self.stored is not None and label in self.stored, f"no stored reference result for {self.case} / {label}"
        return self.stored[label]

    def check(self, label: str, a) -> None:
        import hashlib

        import numpy as np

        exp = self._expected(label)
        a = np.ascontiguousarray(a)
        assert [str(a.dtype), list(a.shape)] == [exp["dtype"], exp["shape"]], (label, a.dtype, a.shape, exp)
        sample = a.reshape(-1)[exp["at"]]
        ref_sample = np.asarray(exp["sample"], dtype=a.dtype)
        assert sample.tobytes() == ref_sample.tobytes(), f"{label}: values {sample} at {exp['at']} != reference {ref_sample}"
        assert hashlib.sha256(a.tobytes()).hexdigest() == exp["sha256"], f"{label}: bits differ from the reference's"

    def check_value(self, label: str, v) -> None:
        assert v == self._expected(label), (label, v, self._expected(label))

    def check_run(self, eng, prefix: str = "") -> None:
        """A finished run(): PI iterations, evaluation sweeps, policy and value-function bits."""
        self.check_value(prefix + "pi_iterations", eng.pi_iterations)
        self.check_value(prefix + "total_sweeps", eng.total_eval_sweeps)
        self.check(prefix + "policy", eng.policy)
        self.check(prefix + "value_function", eng.value_function)


@pytest.fixture()
def reference(request):
    """The reference's results for this test case (see ReferenceGolden)."""
    import json

    case = f"{Path(str(request.node.fspath)).name}::{request.node.nodeid.split('::', 1)[1]}"
    assert REFERENCE_GOLDEN.exists(), f"{REFERENCE_GOLDEN} is missing"
    return ReferenceGolden(case, json.loads(REFERENCE_GOLDEN.read_text())["cases"].get(case))
