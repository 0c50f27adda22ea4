"""
Test fixture: one small "chain of integrators" plugin for every dimensionality D = 1..6.

The engine is dimension-generic, but the shipped environments are 2-, 4- and 6-D only.  Odd D is the only case
whose rows have an odd number of words (W = D + 2), so it is the only case that uses the 4-byte row plane, and
D = 1, 3 and 5 have corner, window and plane geometries of their own.  These plugins give every D an engine whose
transitions a plain numpy float32 loop reproduces bit for bit:

* `step_dynamics` uses explicitly rounded intrinsics only (__fadd_rn, __fsub_rn, __fmul_rn) and no transcendentals,
  so no contraction choice of NVRTC can change a successor, a reward or a termination bit.  `step_numpy` is the same
  arithmetic in numpy float32, operation for operation.
* Dims 0 and 1 are a translation-invariant (position, velocity) pair: pos' = pos + DT * vel, vel' = vel + DT * u.
  No other dimension's update reads dim 0 or dim 1 (dim k >= 2 integrates dim k + 1; the last one integrates -u), so
  states along dim 0 have consecutive successors (x-line windows) and a (dim 0, dim 1) plane sees one successor cell
  of the other dimensions (plane-staged sweep).  At D = 1 the only dimension integrates u.
* The rows contain every kind of row: successors clamped on both sides of every dimension, terminated rows (pushing
  right at full action past the right edge of dim 0), absorbing rows (`_terminal_fn`: a goal box around the origin
  of dims 0 and 1), and exact ties (the action 0.5 appears twice, so its two rows are bit-equal everywhere).
* Grids are ragged, small, include a dimension of 2 bins at D >= 4, and their sizes are not multiples of 32.
  shape[0] is a multiple of 4 with shape[0] / 4 <= 32 (x-line K = 2 and 4); at D >= 4 the (dim 0 x dim 1) plane is
  a multiple of 4 states and at most 1024 (plane-staged sweep).
"""
from __future__ import annotations

import numpy as np

from dynamicprogramming_b200.engine import CudaPIConfig, _CudaPolicyIterationBase

F32 = np.float32

SHAPES = {
    1: (203,),
    2: (12, 37),
    3: (12, 7, 5),
    4: (8, 6, 2, 5),
    5: (12, 7, 2, 5, 3),
    6: (8, 5, 2, 3, 3, 2),
}
# node ranges per dimension: dim 0 [-1, 1], dim 1 [-1.5, 1.5], the others [-1, 1] scaled
RANGES = [(-1.0, 1.0), (-1.5, 1.5), (-1.0, 1.0), (-0.8, 0.9), (-1.2, 1.0), (-0.7, 0.7)]
ACTIONS = np.array([-1.0, -0.25, 0.5, 0.5, 1.0], dtype=F32)   # indices 2 and 3: bit-equal rows, exact ties
TIED_ACTIONS = (2, 3)
DT = "0.3f"                      # not a power of two: the products round
REWARD_W = ["1.0f", "0.5f", "0.25f", "0.25f", "0.25f", "0.25f"]
ACTION_COST = "0.1f"
TERM_X = "1.0f"                  # terminated: pos' > TERM_X while pushing right at full action (u > TERM_U)
TERM_U = "0.75f"
GOAL = (0.15, 0.35)              # absorbing: |pos| <= GOAL[0] (and |vel| <= GOAL[1] at D >= 2)
TERMINAL_VALUE = 2.0
GAMMA = 0.9


def _f(lit: str) -> np.float32:
    return F32(float(lit.rstrip("f")))


def _update(D: int, k: int):
    """(source of dim k's increment, sign): ns_k = s_k +/- DT * source; source is 'u' or a state index."""
    if D == 1:
        return "u", 1
    if k == 0:
        return 1, 1
    if k == 1:
        return "u", 1
    if k + 1 < D:
        return k + 1, 1
    return "u", -1


def dynamics_src(D: int) -> str:
    s = ", ".join(f"float s{k}" for k in range(D))
    ns = ", ".join(f"float* n{k}" for k in range(D))
    body = []
    for k in range(D):
        src, sign = _update(D, k)
        x = "u" if src == "u" else f"s{src}"
        op = "__fadd_rn" if sign > 0 else "__fsub_rn"
        body.append(f"    *n{k} = {op}(s{k}, __fmul_rn({DT}, {x}));")
    body.append("    float r = 0.0f;")
    for k in range(D):
        body.append(f"    r = __fsub_rn(r, __fmul_rn({REWARD_W[k]}, __fmul_rn(s{k}, s{k})));")
    body.append(f"    r = __fsub_rn(r, __fmul_rn({ACTION_COST}, __fmul_rn(u, u)));")
    body.append("    *reward = r;")
    body.append(f"    *terminated = (*n0 > {TERM_X}) && (u > {TERM_U});")
    return ("__device__ void step_dynamics(" + s + ", float u, " + ns + ", float* reward, bool* terminated)\n{\n"
            + "\n".join(body) + "\n}\n")


def step_numpy(states: np.ndarray, u: np.ndarray):
    """`step_dynamics` in numpy float32, operation for operation: (next_states (n, D), reward (n,), terminated (n,))."""
    x = np.asarray(states, dtype=F32)
    u = np.broadcast_to(np.asarray(u, dtype=F32), (len(x),))
    D = x.shape[1]
    dt = _f(DT)
    nx = np.empty_like(x)
    for k in range(D):
        src, sign = _update(D, k)
        inc = (dt * (u if src == "u" else x[:, src])).astype(F32)
        nx[:, k] = (x[:, k] + inc) if sign > 0 else (x[:, k] - inc)
    r = np.zeros(len(x), F32)
    for k in range(D):
        r = (r - (_f(REWARD_W[k]) * (x[:, k] * x[:, k]).astype(F32)).astype(F32)).astype(F32)
    r = (r - (_f(ACTION_COST) * (u * u).astype(F32)).astype(F32)).astype(F32)
    term = (nx[:, 0] > _f(TERM_X)) & (u > _f(TERM_U))
    return nx, r, term


def bins_space(D: int) -> dict:
    return {f"x{k}": np.linspace(RANGES[k][0], RANGES[k][1], n, dtype=F32) for k, n in enumerate(SHAPES[D])}


def terminal_mask(states: np.ndarray) -> np.ndarray:
    goal = np.abs(states[:, 0]) <= GOAL[0]
    if states.shape[1] >= 2:
        goal &= np.abs(states[:, 1]) <= GOAL[1]
    return goal


class ChainIntegrator(_CudaPolicyIterationBase):
    """The D-dimensional plugin (N_DIMS set by `plugin_class`)."""

    def _dynamics_cuda_src(self) -> str:
        return dynamics_src(self.N_DIMS)

    def _terminal_fn(self, states: np.ndarray):
        return terminal_mask(states), TERMINAL_VALUE


_CLASSES: dict = {}


def plugin_class(D: int) -> type:
    if D not in _CLASSES:
        _CLASSES[D] = type(f"ChainIntegrator{D}D", (ChainIntegrator,), {"N_DIMS": D})
    return _CLASSES[D]


def make(D: int, config: CudaPIConfig | None = None, **kwargs):
    cfg = config or CudaPIConfig(gamma=GAMMA, theta=1e-5, max_eval_iter=10_000, max_pi_iter=50)
    return plugin_class(D)(bins_space(D), ACTIONS, cfg, **kwargs)
