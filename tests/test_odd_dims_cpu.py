"""Compile coverage of the odd-dimensional engine paths on a machine without a GPU.

The engine instantiates every kernel for D = 1..6, but the shipped environments are 2-, 4- and 6-D.  These checks
compile, for sm_100a through NVRTC, what an odd-D engine would JIT-compile on the device: the table builder and the
rollout kernels of the chain-of-integrators fixture (tests/fixtures/odd_dims.py) at every D, and the x-line and
plane-staged sweeps at D = 3 and 5 in the configurations their applicability checks accept.  Configurations those
checks reject must be refused with PI_ERR_INVALID before any compile."""
import ctypes as C
import importlib.util
import re
from pathlib import Path

import pytest

from dynamicprogramming_b200 import _ffi

_spec = importlib.util.spec_from_file_location("odd_dims", Path(__file__).resolve().parent / "fixtures" / "odd_dims.py")
odd = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(odd)


def _check(fn, *args) -> int:
    n = C.c_int64()
    _ffi.check(fn(*args, C.byref(n)))
    return n.value


@pytest.mark.parametrize("D", [1, 2, 3, 4, 5, 6])
def test_table_builder_compiles_for_the_fixture(D):
    assert _check(_ffi.lib().pi_compile_check, odd.dynamics_src(D).encode(), D) > 1000


@pytest.mark.parametrize("D", [1, 2, 3, 4, 5, 6])
def test_rollout_kernels_compile_for_the_fixture(D):
    assert _check(_ffi.lib().pi_rollout_compile_check, odd.dynamics_src(D).encode(), D) > 1000


def test_fixture_source_uses_rounded_intrinsics_only():
    """No plain float arithmetic in step_dynamics: nothing NVRTC could contract into an FMA."""
    for D in range(1, 7):
        body = odd.dynamics_src(D).split("{", 1)[1]
        for line in body.splitlines():
            if " = " in line:
                rhs = line.split(" = ", 1)[1].replace("*n0", "")   # the termination test reads the stored *n0
                assert not re.search(r"[-+*/]", rhs), line


# x-line: "K,LV,PF,warps,minb,roll:T..." (one tile size per non-fast position); bins of the synthetic grid per case
XLINE_OK = [(3, 8, "2,0,4,8,2,1:1,8"), (3, 8, "4,0,4,8,1,1:2,4"), (3, 12, "2,0,4,8,2,1:1,12"), (3, 12, "4,0,2,4,1,2:3,4"),
            (5, 8, "2,0,4,8,2,1:1,1,2,4"), (5, 8, "4,0,4,8,1,1:1,1,2,8"), (5, 12, "2,1,4,8,2,2:1,1,1,3"),
            (5, 8, "plane:0,0,2,2,2"), (5, 8, "plane:0,0,2,2,0"), (5, 8, "plane:0,0,2,1,2"), (5, 8, "plane:34,5,2,2,1")]


@pytest.mark.parametrize("D,bins,cfg", XLINE_OK)
def test_odd_dim_jit_sweeps_compile(D, bins, cfg):
    assert _check(_ffi.lib().pi_xline_compile_check, D, bins, cfg.encode()) > 1000


XLINE_REFUSED = [(3, 8, "2,1,4,8,2,4:1,8", "roll"),              # roll 4 needs D >= 4: a D = 3 window has 4 corners
                 (3, 8, "2,0,8,8,2,2:1,8", "PF"),                # PF > windows / roll
                 (3, 10, "4,0,4,8,1,1:1,10", "K"),               # 10 nodes per x-line: not a multiple of K = 4
                 (1, 8, "2,0,4,8,2,1:", "bad argument"),         # the x-line sweep needs D >= 3
                 (3, 8, "plane:0,0,2,2,2", "4 <= D"),            # the plane-staged sweep needs D >= 4
                 (5, 34, "plane:0,0,2,2,2", "1024")]             # a 34 x 34 V-plane is over 1024 states


@pytest.mark.parametrize("D,bins,cfg,why", XLINE_REFUSED)
def test_inapplicable_jit_sweeps_are_refused(D, bins, cfg, why):
    lib = _ffi.lib()
    n = C.c_int64()
    assert lib.pi_xline_compile_check(D, bins, cfg.encode(), C.byref(n)) == _ffi.PI_ERR_INVALID
    assert why in lib.pi_last_error().decode()
