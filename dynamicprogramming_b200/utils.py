"""
GPU counterpart of the reference's inference helpers (utils/barycentric.py):

    get_optimal_action(state, policy, action_space, bounds_low, bounds_high,
                       grid_shape, strides, corner_bits)            utils/barycentric.py:76-108

The reference interpolates ONE state per call on the CPU (numba, single thread); here the
policy table lives on the device and a call answers a whole batch of states with one CUDA
thread each (libdpb200.so: pi_lookup_create / pi_lookup_query, include/dpb200.h).  The
arithmetic of get_barycentric_weights_and_indices (:11-73) is reproduced as numba types it;
the result of a query equals `lambdas @ action_space[policy[flat_indices]]` up to the
summation order of the float32 dot product.  There is no CPU fallback.

PolicyRollout runs what the reference's evaluate() loops over on the CPU — get_optimal_action, then one environment
step — for a batch of episodes on the device, with the plugin's own `step_dynamics` as the simulator
(pi_rollout_create / pi_rollout_run / pi_rollout_step).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _ffi


def _policy_table(policy, action_space, bounds_low, bounds_high, grid_shape):
    """(pi_grid, int32 policy, float32 actions) of a reference-order policy table, as pi_lookup_create and
    pi_rollout_create take them."""
    shape = [int(x) for x in np.asarray(grid_shape).ravel()]
    pol = np.ascontiguousarray(policy, dtype=np.int32).ravel()
    if pol.size != int(np.prod(shape, dtype=np.int64)):
        raise ValueError(f"policy has {pol.size} entries, grid_shape {shape} needs {int(np.prod(shape))}")
    act = np.ascontiguousarray(action_space, dtype=np.float32).ravel()
    grid = _ffi.PiGrid()
    grid.n_dims = len(shape)
    for d in range(len(shape)):
        grid.shape[d] = shape[d]
        grid.lo[d] = float(np.float32(bounds_low[d]))
        grid.hi[d] = float(np.float32(bounds_high[d]))
    return grid, pol, act


class PolicyLookup:
    """Device-resident policy table + batched `get_optimal_action`."""

    def __init__(self, policy: np.ndarray, action_space: np.ndarray, bounds_low: np.ndarray, bounds_high: np.ndarray,
                 grid_shape: np.ndarray, device: int = 0) -> None:
        lib = _ffi.lib()
        grid, pol, act = _policy_table(policy, action_space, bounds_low, bounds_high, grid_shape)
        self.n_dims = grid.n_dims
        handle = C.c_void_p()
        _ffi.check(lib.pi_lookup_create(C.byref(grid), _ffi.ptr(pol), _ffi.ptr(act), len(act), int(device), C.byref(handle)))
        self._h = handle

    def __call__(self, states: np.ndarray) -> np.ndarray:
        """states: (n, D) or (D,) float -> interpolated actions, (n,) float32."""
        pts = np.ascontiguousarray(np.atleast_2d(states), dtype=np.float32)
        if pts.shape[1] != self.n_dims:
            raise ValueError(f"states must have {self.n_dims} columns, got {pts.shape}")
        out = np.empty(len(pts), dtype=np.float32)
        _ffi.check(_ffi.lib().pi_lookup_query(self._h, _ffi.ptr(pts), len(pts), _ffi.ptr(out)))
        return out

    def close(self) -> None:
        if getattr(self, "_h", None):
            _ffi.lib().pi_lookup_destroy(self._h)
            self._h = None

    def __del__(self) -> None:  # pragma: no cover
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass


@dataclass
class RolloutResult:
    """Outputs of PolicyRollout.run for n episodes of up to T steps (episode-major).  The trajectory arrays are None
    unless recorded; their entries after an episode's `length` are NaN."""
    total_reward: np.ndarray        # (n,) float64: sum of r_t
    discounted_return: np.ndarray   # (n,) float64: sum of gamma^t r_t
    length: np.ndarray              # (n,) int32: steps taken
    terminated: np.ndarray          # (n,) bool: step_dynamics set *terminated at the last step
    final_states: np.ndarray        # (n, D) float32: x_length
    states: np.ndarray | None = None    # (n, T+1, D) float32: x_0 .. x_T
    actions: np.ndarray | None = None   # (n, T) float32: a_t
    rewards: np.ndarray | None = None   # (n, T) float32: r_t


class PolicyRollout:
    """Closed-loop rollouts of a policy table under the plugin's own dynamics (include/dpb200.h: pi_rollout_*): the
    loop of the reference's evaluate() — get_optimal_action, then one environment step — for a whole batch of episodes,
    one CUDA thread per episode.  The simulator is the float32 `step_dynamics` the DP was solved with (compiled by
    NVRTC like the table builder), not gymnasium.  `policy` is in reference order (a saved policy's layout)."""

    def __init__(self, policy: np.ndarray, action_space: np.ndarray, bounds_low: np.ndarray, bounds_high: np.ndarray,
                 grid_shape: np.ndarray, dynamics_src: str, device: int = 0) -> None:
        lib = _ffi.lib()
        grid, pol, act = _policy_table(policy, action_space, bounds_low, bounds_high, grid_shape)
        self.n_dims = grid.n_dims
        handle = C.c_void_p()
        _ffi.check(lib.pi_rollout_create(C.byref(grid), _ffi.ptr(pol), _ffi.ptr(act), len(act), dynamics_src.encode(),
                                         int(device), C.byref(handle)))
        self._h = handle

    def _states(self, states: np.ndarray) -> np.ndarray:
        pts = np.ascontiguousarray(np.atleast_2d(states), dtype=np.float32)
        if pts.ndim != 2 or pts.shape[1] != self.n_dims:
            raise ValueError(f"states must have {self.n_dims} columns, got {pts.shape}")
        return pts

    def run(self, initial_states: np.ndarray, n_steps: int, gamma: float, record: bool = False) -> RolloutResult:
        """Episodes from `initial_states` (n, D) for up to `n_steps` steps each; `record` also returns the states,
        actions and rewards of every step."""
        x0 = self._states(initial_states)
        n, D, T = len(x0), self.n_dims, int(n_steps)
        res = RolloutResult(np.empty(n, np.float64), np.empty(n, np.float64), np.empty(n, np.int32),
                            np.empty(n, np.uint8), np.empty((n, D), np.float32))
        traj = [None, None, None]
        if record:
            res.states = np.empty((n, max(T, 0) + 1, D), np.float32)
            res.actions = np.empty((n, max(T, 0)), np.float32)
            res.rewards = np.empty((n, max(T, 0)), np.float32)
            traj = [_ffi.ptr(res.states), _ffi.ptr(res.actions), _ffi.ptr(res.rewards)]
        _ffi.check(_ffi.lib().pi_rollout_run(self._h, _ffi.ptr(x0), n, T, float(gamma), _ffi.ptr(res.total_reward),
                                             _ffi.ptr(res.discounted_return), _ffi.ptr(res.length),
                                             _ffi.ptr(res.terminated), _ffi.ptr(res.final_states), *traj))
        res.terminated = res.terminated.astype(bool)
        return res

    def step(self, states: np.ndarray, actions: np.ndarray) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """One step_dynamics call per (states[i], actions[i]) -> (next_states (n, D) float32, rewards (n,) float32,
        terminated (n,) bool)."""
        x = self._states(states)
        a = np.ascontiguousarray(np.broadcast_to(np.asarray(actions, dtype=np.float32).ravel(), (len(x),)))
        nx = np.empty_like(x)
        r = np.empty(len(x), np.float32)
        t = np.empty(len(x), np.uint8)
        _ffi.check(_ffi.lib().pi_rollout_step(self._h, _ffi.ptr(x), _ffi.ptr(a), len(x), _ffi.ptr(nx), _ffi.ptr(r),
                                              _ffi.ptr(t)))
        return nx, r, t.astype(bool)

    def close(self) -> None:
        if getattr(self, "_h", None):
            _ffi.lib().pi_rollout_destroy(self._h)
            self._h = None

    def __del__(self) -> None:  # pragma: no cover
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass


_cache: dict = {}


def _fingerprint(policy, action_space, bounds_low, bounds_high, grid_shape) -> tuple:
    """Cheap content check of everything the device table was built from: the grid, the action values and a strided
    sample + checksum of the policy (an in-place policy update or a recycled id() must not return stale actions)."""
    pol = np.asarray(policy)
    flat = pol.ravel()
    step = max(1, flat.size // 4096)
    return (tuple(int(x) for x in np.asarray(grid_shape).ravel()),
            np.asarray(bounds_low, dtype=np.float32).tobytes(), np.asarray(bounds_high, dtype=np.float32).tobytes(),
            np.asarray(action_space, dtype=np.float32).tobytes(), flat.size, flat[::step].tobytes(),
            int(flat.sum(dtype=np.int64)))


def invalidate_lookup_cache() -> None:
    """Drop every cached device table of get_optimal_action."""
    while _cache:
        _cache.popitem()[1][3].close()


def get_optimal_action(state, policy, action_space, bounds_low, bounds_high, grid_shape, strides=None, corner_bits=None,
                       device: int | None = None):
    """Drop-in for utils.barycentric.get_optimal_action (same arguments; `strides` and `corner_bits`
    are implied by `grid_shape` and accepted for compatibility).  Accepts one state or a batch.  The device table is
    cached per (policy, action_space) object pair and revalidated on every call against a fingerprint of the policy,
    the action values and the grid; `device` defaults to LOCAL_RANK (0 outside torchrun)."""
    import os

    dev = int(os.environ.get("LOCAL_RANK", 0)) if device is None else int(device)
    key = (id(policy), id(action_space), dev)
    fp = _fingerprint(policy, action_space, bounds_low, bounds_high, grid_shape)
    hit = _cache.get(key)
    if hit is None or hit[0] is not policy or hit[1] is not action_space or hit[2] != fp:
        if hit is not None:
            _cache.pop(key)[3].close()
        if len(_cache) >= 4:
            _cache.pop(next(iter(_cache)))[3].close()
        hit = (policy, action_space, fp, PolicyLookup(policy, action_space, bounds_low, bounds_high, grid_shape, device=dev))
        _cache[key] = hit
    out = hit[3](state)
    return out[0] if np.ndim(state) == 1 else out
