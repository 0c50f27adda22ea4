"""
Host-side mirror of the reference's engine interface
(src/cuda_policy_iteration.py of nicoRomeroCuruchet/DynamicProgramming):

    CudaPIConfig                        :36-43
    CudaPolicyIteration2D / 4D / 6D     :46, :439, :847

Same constructor, same abstract plugin hooks (`_dynamics_cuda_src`,
`_terminal_fn`), same methods (`policy_evaluation`, `policy_improvement`,
`run`, `save`, `load`) and the same public attributes, so an environment class
written for the reference subclasses these unchanged.  Underneath, every
method is a call into libdpb200.so (hand-written sm_100a CUDA behind the C ABI
of include/dpb200.h).  There is no CPU path: constructing an engine without a
CUDA device raises RuntimeError, like the reference does without cupy (:71-75).
"""
from __future__ import annotations

import abc
import ctypes as C
import os
from dataclasses import dataclass
from itertools import product
from pathlib import Path

import numpy as np

from . import _ffi

try:  # the reference logs through loguru; keep the same sink when present
    from loguru import logger
except ImportError:  # pragma: no cover
    import logging

    class _Shim:
        _l = logging.getLogger("dynamicprogramming_b200")

        def debug(self, m): self._l.debug(m)
        def info(self, m): self._l.info(m)
        def success(self, m): self._l.info(m)
        def warning(self, m): self._l.warning(m)

    logger = _Shim()


@dataclass
class CudaPIConfig:
    """Same fields and defaults as the reference (src/cuda_policy_iteration.py:36-43)."""
    gamma: float = 0.99
    theta: float = 1e-4
    max_eval_iter: int = 10_000
    max_pi_iter: int = 50
    log_interval: int = 100


# ── N4: engines kept alive across trainings ──────────────────────────────────────────────────────────────────────
# The autoresearch loop of the reference (runners/trial_runner.sh:33-60) trains the same grid again and again with an
# edited dynamics / reward string.  With keep_engines(True) (or DPB200_KEEP_ENGINE=1) `close()` parks the native engine
# instead of destroying it, and the next constructor call for the SAME grid, action set, config, device and shard takes
# it over through pi_retrain: CUDA context, buffers, storage order, JIT sweep kernels, graphs and communicator are
# reused; only the table builder is recompiled (when the text changed) and the table rebuilt.
_KEEP_ENGINES = os.environ.get("DPB200_KEEP_ENGINE", "0") not in ("0", "", "off")
_ENGINE_POOL: dict = {}


def keep_engines(on: bool = True) -> None:
    """Enable / disable parking of native engines on close() (see above); disabling releases the parked ones."""
    global _KEEP_ENGINES
    _KEEP_ENGINES = bool(on)
    if not on:
        release_engines()


def release_engines() -> None:
    """Destroy every parked engine (frees its VRAM)."""
    while _ENGINE_POOL:
        _, handle = _ENGINE_POOL.popitem()
        _ffi.lib().pi_destroy(handle)


# states above which `_terminal_fn` is evaluated slab by slab instead of on the
# fully materialised (N, D) array (host memory / time; results are identical
# for the element-wise masks every reference environment uses).
_CHUNK_STATES = int(os.environ.get("DPB200_TERMINAL_CHUNK", 2_000_000))
# ... unless the plugin stashes per-state arrays inside `_terminal_fn`: up to this size it then gets the whole grid in one
# call (the reference's behaviour); above it the stashed slabs are stitched (host memory: N x D x 4 bytes)
_FULL_STATES_MAX = 16_000_000


class DeviceArray:
    """Non-owning handle on an engine device buffer (the `d_*` attributes of the
    reference object).  Exposes __cuda_array_interface__ so torch / cupy can
    wrap it zero-copy: ``torch.as_tensor(pi.d_value_function, device="cuda")``."""

    def __init__(self, ptr: int, shape: tuple, typestr: str, owner, role: int | None = None) -> None:
        self._ptr, self.shape, self._typestr, self._owner, self._role = ptr, shape, typestr, owner, role

    def __setitem__(self, key, value) -> None:
        """``d_value_function[mask] = scalar`` with a boolean mask over the whole grid in reference
        order — the store a reference subclass does on its cupy arrays
        (runners/overhead_crane_cuda.py:199-202).  The buffer itself is in the engine's storage
        order, so the store goes through pi_set_values_buffer rather than raw indexing."""
        if self._role is None:
            raise TypeError("this device buffer is read-only from Python")
        if hasattr(key, "get"):          # a cupy array
            key = key.get()
        mask = np.asarray(key)
        if mask.dtype != np.bool_ or mask.shape != (self._owner.n_states,):
            raise TypeError("only boolean-mask stores over the whole grid (n_states,) are supported")
        m = np.ascontiguousarray(mask, dtype=np.uint8)
        _ffi.check(_ffi.lib().pi_set_values_buffer(self._owner._engine, self._role, _ffi.ptr(m), float(value)))

    @property
    def __cuda_array_interface__(self) -> dict:
        return {"shape": self.shape, "typestr": self._typestr, "data": (self._ptr, False), "version": 3,
                "strides": None}

    def torch(self):
        import torch
        return torch.as_tensor(self, device=f"cuda:{self._owner._device}")

    def raw(self) -> np.ndarray:
        """The buffer as the engine stores it (internal storage order, see `layout()`)."""
        return self.torch().cpu().numpy()

    def get(self) -> np.ndarray:
        """Host copy in REFERENCE order — what `cupy_array.get()` returns on the reference object.  The engine may
        store states with other dimensions fastest (pi_layout); full-grid buffers are put back into reference order
        here, shard-local buffers of a sharded run cannot be and raise."""
        a = self.raw()
        eng = self._owner
        perm = eng.layout()["perm"]
        if perm == list(range(eng.N_DIMS)):
            return a
        if a.shape != (eng.n_states,):
            raise RuntimeError("this buffer holds one shard in the engine's storage order; use download() for reference order")
        shape_int = [int(eng.grid_shape[d]) for d in perm]
        inv = [perm.index(d) for d in range(eng.N_DIMS)]
        return np.ascontiguousarray(a.reshape(shape_int).transpose(inv)).ravel()


class _CudaPolicyIterationBase(abc.ABC):
    """Dimension-generic implementation behind the 2D/4D/6D classes."""

    N_DIMS: int = 0

    def __init__(self, bins_space: dict, action_space: np.ndarray, config: CudaPIConfig | None = None,
                 *, device: int | None = None, shard: tuple | None = None) -> None:
        _ffi.lib()  # raises if the CUDA extension is missing
        self.config = config or CudaPIConfig()
        self.action_space = np.ascontiguousarray(action_space, dtype=np.float32)
        self.n_actions = len(self.action_space)

        keys = list(bins_space.keys())
        assert len(keys) == self.N_DIMS, (
            f"CudaPolicyIteration{self.N_DIMS}D requires exactly {self.N_DIMS} state dimensions."
        )
        # per-axis node coordinates: the float32 bits the reference stores in states_space columns
        self._axes = [np.ascontiguousarray(np.asarray(bins_space[k]).astype(np.float32)) for k in keys]
        self._axis_names = keys
        self.n_states = int(np.prod([len(a) for a in self._axes], dtype=np.int64))
        self._states_space = None
        self._device = int(os.environ.get("LOCAL_RANK", 0)) if device is None else int(device)
        self._shard = shard  # (rank, world_size, nccl_id bytes)
        self._engine = None
        self._table_ready = False
        self._log_cb = None

        self._precompute_grid_metadata()
        self._allocate_tensors_and_compile()

    # ── Grid metadata (src/cuda_policy_iteration.py:95-109, :497-514, :912-937) ──

    @property
    def states_space(self) -> np.ndarray:
        """(n_states, D) float32, row-major, dim 0 slowest — materialised on first use
        (the reference builds it eagerly with meshgrid(indexing="ij") + column_stack)."""
        if self._states_space is None:
            if getattr(self, "_axes", None) is not None:
                grids = np.meshgrid(*self._axes, indexing="ij")
                self._states_space = np.column_stack([g.ravel() for g in grids]).astype(np.float32)
            else:   # an instance made by load(): read the entry now
                with np.load(self._states_file) as data:
                    self._states_space = data["states_space"]
        return self._states_space

    @states_space.setter
    def states_space(self, value) -> None:
        self._states_space = value

    def _precompute_grid_metadata(self) -> None:
        D = self.N_DIMS
        # min / max / unique over a column of the meshgrid equal the same over its axis
        self.bounds_low = np.array([a.min() for a in self._axes], dtype=np.float32)
        self.bounds_high = np.array([a.max() for a in self._axes], dtype=np.float32)
        self.grid_shape = np.array([len(np.unique(a)) for a in self._axes], dtype=np.int32)
        for d, a in enumerate(self._axes):
            if self.grid_shape[d] != len(a):
                raise ValueError(f"bins_space[{self._axis_names[d]!r}] contains duplicate nodes")
        strides = np.ones(D, dtype=np.int64)
        for d in range(D - 2, -1, -1):
            strides[d] = strides[d + 1] * self.grid_shape[d + 1]
        self.strides = strides.astype(np.int32)
        self.corner_bits = np.array(list(product([0, 1], repeat=D)), dtype=np.int32)
        logger.info(f"Grid: shape={self.grid_shape.tolist()}, states={self.n_states:,}, actions={self.n_actions}")

    # ── Plugin interface (identical to the reference) ─────────────────────────

    @abc.abstractmethod
    def _dynamics_cuda_src(self) -> str:
        """CUDA source defining
            __device__ void step_dynamics(float s0, ..., float s{D-1}, float action,
                                          float* ns0, ..., float* ns{D-1},
                                          float* reward, bool* terminated)
        (src/cuda_policy_iteration.py:113-125, :518-530, :941-954)."""

    def _terminal_fn(self, states: np.ndarray) -> tuple[np.ndarray, float]:
        """(bool mask over states, terminal value); default: none (:127-138)."""
        return np.zeros(len(states), dtype=bool), 0.0

    # ── Device allocation & compilation (:142-175) ─────────────────────────────

    def _terminal_mask_and_value(self) -> tuple[np.ndarray, float]:
        if type(self)._terminal_fn is _CudaPolicyIterationBase._terminal_fn:
            return np.zeros(self.n_states, dtype=bool), 0.0
        if self.n_states <= _CHUNK_STATES:
            mask, value = self._terminal_fn(self.states_space)
            return np.asarray(mask, dtype=bool), float(value)
        # slab-wise over dim 0
        inner = self.n_states // len(self._axes[0])
        chunk = np.empty((inner, self.N_DIMS), dtype=np.float32)   # one slab buffer: only column 0 changes
        for d, g in enumerate(np.meshgrid(*self._axes[1:], indexing="ij")):
            chunk[:, d + 1] = g.ravel()
        mask = np.empty(self.n_states, dtype=bool)
        value = 0.0
        # per-state arrays a plugin stashes on itself inside _terminal_fn (the crane's `_goal_mask`,
        # runners/overhead_crane_cuda.py:189) are stitched back together over the slabs
        stashed: dict[str, list] = {}
        for i, x0 in enumerate(self._axes[0]):
            chunk[:, 0] = x0
            before = {k: id(v) for k, v in vars(self).items()}
            m, value = self._terminal_fn(chunk)
            mask[i * inner:(i + 1) * inner] = m
            for k, v in vars(self).items():
                if isinstance(v, np.ndarray) and v.shape[:1] == (inner,) and before.get(k) != id(v):
                    stashed.setdefault(k, []).append(v.copy())
            if i == 0 and stashed and self.n_states <= _FULL_STATES_MAX:
                # the plugin keeps per-state arrays from _terminal_fn (the crane's goal mask): give it the whole grid at once,
                # exactly as the reference does, instead of stitching slabs back together
                mask, value = self._terminal_fn(self.states_space)
                return np.asarray(mask, dtype=bool), float(value)
        for k, parts in stashed.items():
            if len(parts) == len(self._axes[0]):
                setattr(self, k, np.concatenate(parts))
        return mask, float(value)

    def _allocate_tensors_and_compile(self) -> None:
        logger.info("Allocating GPU tensors and compiling CUDA kernels...")
        lib = _ffi.lib()
        D = self.N_DIMS
        grid = _ffi.PiGrid()
        grid.n_dims = D
        for d in range(D):
            grid.shape[d] = int(self.grid_shape[d])
            grid.lo[d] = float(self.bounds_low[d])
            grid.hi[d] = float(self.bounds_high[d])
            grid.axes[d] = self._axes[d].ctypes.data_as(C.POINTER(C.c_float))
        cfg = _ffi.PiConfig(float(self.config.gamma), float(self.config.theta), int(self.config.max_eval_iter),
                            int(self.config.max_pi_iter), int(self.config.log_interval), 25)
        shard_p = None
        if self._shard is not None and self._shard[1] > 1:
            sh = _ffi.PiShard()
            sh.rank, sh.world_size = int(self._shard[0]), int(self._shard[1])
            C.memmove(sh.nccl_id, bytes(self._shard[2]), 128)
            shard_p = C.byref(sh)
        self._pool_key = None
        if self._shard is None or self._shard[1] <= 1:
            self._pool_key = (D, tuple(a.tobytes() for a in self._axes), self.action_space.tobytes(),
                              (cfg.gamma, cfg.theta, cfg.max_eval_iter, cfg.max_pi_iter, cfg.log_interval), self._device)
        handle = _ENGINE_POOL.pop(self._pool_key, None) if _KEEP_ENGINES and self._pool_key is not None else None
        reused = handle is not None
        if not reused:
            handle = C.c_void_p()
            _ffi.check(lib.pi_create(C.byref(grid), self.action_space.ctypes.data_as(C.POINTER(C.c_float)),
                                     self.n_actions, C.byref(cfg), self._dynamics_cuda_src().encode(), self._device,
                                     shard_p, C.byref(handle)))
        self._engine = handle

        levels = {0: logger.debug, 1: logger.info, 2: logger.success, 3: logger.warning}
        self._log_cb = _ffi.LOG_FN(lambda lvl, msg, _u: levels.get(lvl, logger.info)(msg.decode(errors="replace")))
        _ffi.check(lib.pi_set_log(self._engine, self._log_cb, None))

        terminal_mask, terminal_value = self._terminal_mask_and_value()
        self._terminal_mask_host = np.ascontiguousarray(terminal_mask, dtype=np.uint8)
        has_terminal = bool(self._terminal_mask_host.any())
        if reused:
            self._retrain_native(has_terminal, terminal_value)
        elif has_terminal:
            _ffi.check(lib.pi_set_terminal(self._engine, _ffi.ptr(self._terminal_mask_host), float(terminal_value)))
        if has_terminal:
            logger.info(f"Terminal states: {int(terminal_mask.sum()):,} (value={terminal_value})")
        self._refresh_device_handles()
        logger.success("CUDA kernels compiled. VRAM allocated.")

    def _retrain_native(self, has_terminal: bool, terminal_value: float) -> bool:
        """pi_retrain with this object's current dynamics text and terminal mask; True if the builder was recompiled."""
        recompiled = C.c_int32()
        mask = _ffi.ptr(self._terminal_mask_host) if has_terminal else None
        _ffi.check(_ffi.lib().pi_retrain(self._engine, self._dynamics_cuda_src().encode(), mask, float(terminal_value),
                                         C.byref(recompiled)))
        self._table_ready = True
        return bool(recompiled.value)

    def retrain(self) -> bool:
        """In-process counterpart of a new trial: re-read `_dynamics_cuda_src()` / `_terminal_fn` from this object (a
        subclass instance whose reward or dynamics parameters were edited), rebuild the transition table and reset V
        and the policy — keeping the CUDA context, buffers, JIT sweep kernels, graphs and communicator
        (include/dpb200.h: pi_retrain).  Returns True if the dynamics text changed and was recompiled.  Follow with
        policy_evaluation() / policy_improvement() or run()."""
        terminal_mask, terminal_value = self._terminal_mask_and_value()
        self._terminal_mask_host = np.ascontiguousarray(terminal_mask, dtype=np.uint8)
        out = self._retrain_native(bool(self._terminal_mask_host.any()), terminal_value)
        self._refresh_device_handles()
        return out

    def _refresh_device_handles(self) -> None:
        lib = _ffi.lib()
        v, nv, pol, term = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        _ffi.check(lib.pi_device_ptrs(self._engine, C.byref(v), C.byref(nv), C.byref(pol), C.byref(term)))
        n_local = lib.pi_local_end(self._engine) - lib.pi_local_begin(self._engine)
        self.d_value_function = DeviceArray(v.value, (self.n_states,), "<f4", self, role=0)
        self.d_new_value_function = DeviceArray(nv.value, (self.n_states,), "<f4", self, role=1)
        self.d_policy = DeviceArray(pol.value, (n_local,), "<i4", self)
        self.d_terminal_mask = DeviceArray(term.value, (n_local,), "|u1", self)

    def set_values(self, mask: np.ndarray, value: float) -> None:
        """V[mask] = value on both buffers (the crane's goal initialisation,
        runners/overhead_crane_cuda.py:193-206)."""
        m = np.ascontiguousarray(mask, dtype=np.uint8)
        _ffi.check(_ffi.lib().pi_set_values(self._engine, _ffi.ptr(m), float(value)))

    def build_table(self) -> None:
        """Transition-table build (new stage; runs once, before the first sweep)."""
        if not self._table_ready:
            _ffi.check(_ffi.lib().pi_build_table(self._engine))
            self._table_ready = True

    # ── Policy iteration (:300-370) ───────────────────────────────────────────

    def policy_evaluation(self) -> float:
        """Iterative policy evaluation until convergence; returns the last residual."""
        self.build_table()
        delta, sweeps = C.c_float(), C.c_int32()
        _ffi.check(_ffi.lib().pi_evaluate(self._engine, C.byref(delta), C.byref(sweeps)))
        self.last_eval_sweeps = int(sweeps.value)
        self._refresh_device_handles()
        return float(delta.value)

    def policy_improvement(self) -> bool:
        """Greedy improvement; True if the policy is stable."""
        self.build_table()
        stable, changed = C.c_int32(), C.c_int64()
        _ffi.check(_ffi.lib().pi_improve(self._engine, C.byref(stable), C.byref(changed)))
        self.last_changed = int(changed.value)
        return bool(stable.value)

    def run(self) -> None:
        """The complete policy-iteration loop (same for/else semantics as :357-370)."""
        self.total_eval_sweeps = 0
        self.pi_iterations = 0
        self.converged = False
        for n in range(self.config.max_pi_iter):
            logger.info(f"-- PI Iteration {n + 1}/{self.config.max_pi_iter} --")
            self.policy_evaluation()
            self.total_eval_sweeps += self.last_eval_sweeps
            self.pi_iterations = n + 1
            if self.policy_improvement():
                self.converged = True
                logger.success(f"Policy Iteration converged at iteration {n + 1}.")
                break
        else:
            logger.warning(f"Policy Iteration hit max_pi_iter={self.config.max_pi_iter}.")
        self._pull_tensors_from_gpu()

    def engine_stats(self) -> dict:
        st = _ffi.PiStats()
        _ffi.check(_ffi.lib().pi_get_stats(self._engine, C.byref(st)))
        d = st.as_dict()
        d["launches"] = int(_ffi.lib().pi_launch_count(self._engine))
        d["table_bytes"] = int(_ffi.lib().pi_table_bytes(self._engine))
        return d

    def _pull_tensors_from_gpu(self) -> None:
        """D2H of V and policy, then release VRAM (:372-388)."""
        logger.info("Pulling results from VRAM to RAM...")
        self.value_function = np.empty(self.n_states, dtype=np.float32)
        self.policy = np.empty(self.n_states, dtype=np.int32)
        _ffi.check(_ffi.lib().pi_copy_results(self._engine, _ffi.ptr(self.value_function), _ffi.ptr(self.policy)))
        self.stats = self.engine_stats()
        self.close()
        logger.success("VRAM released. Results in CPU RAM.")

    def close(self) -> None:
        if getattr(self, "_engine", None):
            key = getattr(self, "_pool_key", None)
            if _KEEP_ENGINES and key is not None and key not in _ENGINE_POOL and len(_ENGINE_POOL) < 2:
                _ffi.lib().pi_set_log(self._engine, _ffi.LOG_FN(0), None)   # the callback dies with this object
                _ENGINE_POOL[key] = self._engine                           # parked: the next constructor for this grid retrains it
            else:
                _ffi.lib().pi_destroy(self._engine)
            self._engine = None
            for attr in ("d_value_function", "d_new_value_function", "d_policy", "d_terminal_mask"):
                if hasattr(self, attr):
                    delattr(self, attr)

    def __del__(self) -> None:  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    # ── Persistence: the reference's nine-array .npz (:392-432) ───────────────

    def save(self, filepath: Path | str) -> None:
        """The reference's nine-array uncompressed .npz (:392-409), same keys, dtypes, shapes and order.
        `states_space` (N x D float32: 1.5 GB at 6-D / 20 bins) is the only large entry; when it has
        never been materialised it is STREAMED into the archive slab by slab along dim 0 (SURVEY §8f N3)
        — the file np.load sees is the one np.savez would have written."""
        filepath = Path(filepath).with_suffix(".npz")
        filepath.parent.mkdir(parents=True, exist_ok=True)
        small = dict(
            value_function=self.value_function,
            policy=self.policy,
            bounds_low=self.bounds_low,
            bounds_high=self.bounds_high,
            grid_shape=self.grid_shape,
            strides=self.strides,
            corner_bits=self.corner_bits,
            action_space=self.action_space,
        )
        if self._states_space is not None or getattr(self, "_axes", None) is None:
            np.savez(filepath, **small, states_space=self.states_space)
        else:
            self._save_streamed(filepath, small)
        logger.success(f"Policy saved to {filepath.resolve()}")

    def _save_streamed(self, filepath: Path, small: dict) -> None:
        import zipfile

        from numpy.lib import format as npy_format

        D = self.N_DIMS
        inner = self.n_states // len(self._axes[0])
        with zipfile.ZipFile(filepath, mode="w", compression=zipfile.ZIP_STORED, allowZip64=True) as zf:
            for key, val in small.items():
                with zf.open(key + ".npy", "w", force_zip64=True) as fid:
                    npy_format.write_array(fid, np.asanyarray(val), allow_pickle=False)
            with zf.open("states_space.npy", "w", force_zip64=True) as fid:
                header = {"descr": npy_format.dtype_to_descr(np.dtype(np.float32)), "fortran_order": False,
                          "shape": (self.n_states, D)}
                npy_format.write_array_header_1_0(fid, header)
                if D == 1:
                    fid.write(np.ascontiguousarray(self._axes[0], np.float32).reshape(-1, 1).tobytes())
                else:
                    rest = np.meshgrid(*self._axes[1:], indexing="ij")
                    slab = np.empty((inner, D), dtype=np.float32)
                    for d, g in enumerate(rest):
                        slab[:, d + 1] = g.ravel()
                    del rest
                    for x0 in self._axes[0]:
                        slab[:, 0] = x0
                        fid.write(memoryview(slab).cast("B"))

    @classmethod
    def load(cls, filepath: Path | str):
        """Load a saved policy (no GPU required).  `states_space` is read from the archive on first
        use (np.load is lazy per key), everything else eagerly as the reference does (:411-432)."""
        filepath = Path(filepath).with_suffix(".npz")
        data = np.load(filepath)
        instance = cls.__new__(cls)
        instance._engine = None
        instance._states_space = None
        instance._states_file = filepath
        instance.value_function = data["value_function"]
        instance.policy = data["policy"]
        instance.bounds_low = data["bounds_low"]
        instance.bounds_high = data["bounds_high"]
        instance.grid_shape = data["grid_shape"]
        instance.strides = data["strides"]
        instance.corner_bits = data["corner_bits"]
        instance.action_space = data["action_space"]
        if "states_space" not in data.files:
            raise KeyError("states_space is not a file in the archive")
        instance.n_actions = len(instance.action_space)
        instance.n_states = len(instance.policy)
        instance.config = CudaPIConfig()
        data.close()
        logger.success(f"Policy loaded from {filepath.resolve()}")
        return instance

    # ── Extras beyond the reference surface (tests / bench / e2e call) ─────────

    def upload_policy(self, policy: np.ndarray) -> None:
        self.build_table()
        p = np.ascontiguousarray(policy, dtype=np.int32)
        assert p.shape == (self.n_states,)
        _ffi.check(_ffi.lib().pi_upload_policy(self._engine, _ffi.ptr(p)))

    def upload_policy_local(self, policy_local: np.ndarray) -> None:
        """This rank's slice of the policy in the engine's storage order (see `to_internal_order`,
        `pi_copy_local_results`): no full-grid staging, no collective."""
        p = np.ascontiguousarray(policy_local, dtype=np.int32)
        _ffi.check(_ffi.lib().pi_upload_policy_local(self._engine, _ffi.ptr(p)))

    def upload_values(self, values: np.ndarray) -> None:
        v = np.ascontiguousarray(values, dtype=np.float32)
        assert v.shape == (self.n_states,)
        _ffi.check(_ffi.lib().pi_upload_values(self._engine, _ffi.ptr(v)))

    def warm_start(self, source) -> dict:
        """Start from another grid's solution instead of V = 0, policy = 0 (include/dpb200.h: pi_prolong_values).

        `source` is a saved-policy .npz path, an instance after run() or load() (`value_function`, `bounds_low`,
        `bounds_high`, `grid_shape`), or a `(values, bounds_low, bounds_high, grid_shape)` tuple; its grid is taken as
        uniform.  Every non-absorbing state gets the source V interpolated at its node (clamped to the source box, the
        arithmetic of lookup_actions); absorbing states keep their values.  Then one policy_improvement() makes the
        policy greedy with respect to that V, and a following run() evaluates it starting from the prolonged V.
        Returns {"prolong_ms": device time of the prolongation kernel, "changed": states whose action differs from the
        policy held before (pi = 0 on a fresh engine)}.  retrain() resets V and the policy as usual."""
        values, lo, hi, shape = _warm_start_source(source)
        self.build_table()
        grid = _ffi.PiGrid()
        grid.n_dims = len(shape)
        for d in range(len(shape)):
            grid.shape[d], grid.lo[d], grid.hi[d] = int(shape[d]), float(lo[d]), float(hi[d])
        ms = C.c_float()
        _ffi.check(_ffi.lib().pi_prolong_values(self._engine, C.byref(grid), _ffi.ptr(values), C.byref(ms)))
        self.policy_improvement()
        return {"prolong_ms": float(ms.value), "changed": self.last_changed}

    def download(self, values: np.ndarray | None = None, policy: np.ndarray | None = None):
        if values is None:
            values = np.empty(self.n_states, dtype=np.float32)
        if policy is None:
            policy = np.empty(self.n_states, dtype=np.int32)
        _ffi.check(_ffi.lib().pi_copy_results(self._engine, _ffi.ptr(values), _ffi.ptr(policy)))
        return values, policy

    def sweeps(self, n: int) -> tuple[float, float]:
        """Exactly n evaluation sweeps, no convergence test -> (last residual, device ms)."""
        self.build_table()
        delta, ms = C.c_float(), C.c_float()
        _ffi.check(_ffi.lib().pi_sweeps(self._engine, int(n), C.byref(delta), C.byref(ms)))
        self._refresh_device_handles()
        return float(delta.value), float(ms.value)

    def layout(self) -> dict:
        """Internal storage order chosen by the engine (include/dpb200.h: pi_layout).
        Host-facing arrays are always in reference order; only the raw device
        handles (d_value_function, ...) are stored with `fast_dim` contiguous."""
        fast = C.c_int32()
        perm = (C.c_int32 * _ffi.PI_MAX_DIMS)()
        lines = (C.c_double * _ffi.PI_MAX_DIMS)()
        _ffi.check(_ffi.lib().pi_layout(self._engine, C.byref(fast), perm, lines))
        D = self.N_DIMS
        p = [int(perm[k]) for k in range(D)]
        # two fast dimensions (a "plane" layout for the plane-staged sweep) when the slower ones are not in logical order
        rest = [d for d in range(D) if d != p[-1]]
        return {"fast_dim": int(fast.value), "fast_dim2": p[-2] if D >= 2 and p[:-1] != rest else -1, "perm": p,
                "probe_lines": [float(lines[d]) for d in range(D)]}

    def lookup_actions(self, states: np.ndarray) -> np.ndarray:
        """Batched get_optimal_action (utils/barycentric.py:76-108) for `states` (n, D): on a live engine
        the device-resident policy answers (pi_lookup_actions); after run() / load() the host `policy`
        array is uploaded once into a lookup table (pi_lookup_create)."""
        pts = np.ascontiguousarray(np.atleast_2d(states), dtype=np.float32)
        if pts.shape[1] != self.N_DIMS:
            raise ValueError(f"states must have {self.N_DIMS} columns, got {pts.shape}")
        if getattr(self, "_engine", None):
            out = np.empty(len(pts), dtype=np.float32)
            _ffi.check(_ffi.lib().pi_lookup_actions(self._engine, _ffi.ptr(pts), len(pts), _ffi.ptr(out)))
            return out
        from .utils import PolicyLookup
        look = getattr(self, "_lookup", None)
        if look is None or look[0] is not self.policy:
            if look is not None:
                look[1].close()
            look = (self.policy, PolicyLookup(self.policy, self.action_space, self.bounds_low, self.bounds_high, self.grid_shape,
                                              device=int(getattr(self, "_device", os.environ.get("LOCAL_RANK", 0)))))
            self._lookup = look
        return look[1](pts)

    def _rollout_handle(self, need_current_policy: bool = True):
        """The cached PolicyRollout of this object (see rollout()); rebuilt when the policy object or the dynamics text
        changes.  A live engine's policy is taken through download(); an unchanged download reuses the handle.  A single
        step does not use the policy (need_current_policy=False): any handle built from the same text serves it."""
        from .utils import PolicyRollout
        src = self._dynamics_cuda_src()
        cached = getattr(self, "_rollout", None)
        live = bool(getattr(self, "_engine", None))
        if cached is not None and cached[1] == src and not need_current_policy:
            return cached[2]
        policy = self.download()[1] if live else self.policy
        if cached is not None and cached[1] == src and (cached[0] is policy or (live and np.array_equal(cached[0], policy))):
            return cached[2]
        if cached is not None:
            cached[2].close()
            self._rollout = None
        h = PolicyRollout(policy, self.action_space, self.bounds_low, self.bounds_high, self.grid_shape, src,
                          device=int(getattr(self, "_device", os.environ.get("LOCAL_RANK", 0))))
        self._rollout = (policy, src, h)
        return h

    def rollout(self, initial_states: np.ndarray, n_steps: int, gamma: float | None = None, record: bool = False):
        """Closed-loop episodes of the current policy under this plugin's own `step_dynamics` (what the reference's
        evaluate() does with get_optimal_action + an environment step, batched on the device: utils.PolicyRollout).
        `initial_states` (n, D); each episode runs `n_steps` steps or until step_dynamics sets *terminated.  Works
        after run() and after load() (host `policy`) and on a live engine (its current policy, through download()).
        `gamma=None` is the engine's gamma as float32 (`self.config.gamma`); an instance made by load() carries the
        default CudaPIConfig(), so pass its gamma explicitly there.  Returns a utils.RolloutResult."""
        if gamma is None:
            gamma = float(np.float32(self.config.gamma))
        return self._rollout_handle().run(initial_states, n_steps, gamma, record=record)

    def simulate_step(self, states: np.ndarray, actions: np.ndarray):
        """One step of this plugin's `step_dynamics` per (states[i], actions[i]) on the device ->
        (next_states (n, D) float32, rewards (n,) float32, terminated (n,) bool)."""
        return self._rollout_handle(need_current_policy=False).step(states, actions)

    def eval_kernel_info(self) -> dict:
        """Which evaluation-sweep kernel the build-time autotune selected (include/dpb200.h:
        pi_eval_kernel_info): the scalar gather sweep or the JIT-compiled x-line sweep."""
        buf = C.create_string_buffer(256)
        ms_s, ms_x = C.c_double(), C.c_double()
        kind = _ffi.lib().pi_eval_kernel_info(self._engine, buf, 256, C.byref(ms_s), C.byref(ms_x))
        return {"xline": kind == 1, "plane": kind == 2, "kernel": buf.value.decode(), "probe_ms_scalar": ms_s.value,
                "probe_ms_selected": ms_x.value}

    def debug_plane(self, cfg: str = "", iters: int = 5) -> dict:
        """Test hook: the plane-staged sweep configuration `cfg` ("NS,L,minb,lv,pack", 0 = default) vs the kernel
        the engine currently runs, on the current rows and V; timings, plan statistics and the number of
        differing V words (must be 0)."""
        ms_new, ms_base = C.c_float(), C.c_float()
        mism, st, info = C.c_int64(), (C.c_double * 8)(), (C.c_int32 * 6)()
        _ffi.check(_ffi.lib().pi_debug_plane(self._engine, cfg.encode(), int(iters), C.byref(ms_new), C.byref(ms_base),
                                             C.byref(mism), st, info))
        return {"ms_plane": ms_new.value, "ms_base": ms_base.value, "mismatches": int(mism.value),
                "loads_per_plane": st[0], "late_per_plane": st[1], "cells_per_plane": st[2], "fallback_frac": st[3],
                "pairs_per_plane": st[4], "stray_pairs_per_plane": st[5], "singles_paired_per_plane": st[6], "registers": int(info[0]), "grid": int(info[1]), "block": int(info[2]), "smem": int(info[3]),
                "slots": int(info[4]), "chunk": int(info[5])}

    def debug_xline(self, cfg: str, iters: int = 5) -> dict:
        """Test hook: run the x-line sweep configuration `cfg` and the scalar sweep on the current
        rows and V; returns timings and the number of differing V words (must be 0)."""
        ms_new, ms_base = C.c_float(), C.c_float()
        mism, wf, info = C.c_int64(), C.c_double(), (C.c_int32 * 4)()
        _ffi.check(_ffi.lib().pi_debug_xline(self._engine, cfg.encode(), int(iters), C.byref(ms_new), C.byref(ms_base),
                                             C.byref(mism), C.byref(wf), info))
        return {"ms_xline": ms_new.value, "ms_scalar": ms_base.value, "mismatches": int(mism.value),
                "window_fraction": wf.value, "registers": int(info[0]), "grid": int(info[1]), "block": int(info[2])}

    def debug_pair(self, threads: int = 256, minb: int = 2, iters: int = 5, lv: int = 1, group: int = 0,
                   single: int = 0) -> dict:
        """Test hook: a JIT sweep configuration (csrc/pair_sweep_src.cuh; single = 0 packed pairs, 1 one state per
        thread, 2 one state per thread gathering from the pair shadow of V) vs the scalar sweep (bitwise
        comparison + timings)."""
        ms_p, ms_s, mism, regs = C.c_float(), C.c_float(), C.c_int64(), C.c_int32()
        _ffi.check(_ffi.lib().pi_debug_pair(self._engine, int(threads), int(minb), int(lv), int(group), int(single),
                                            int(iters), C.byref(ms_p), C.byref(ms_s), C.byref(mism), C.byref(regs)))
        return {"ms_pair": ms_p.value, "ms_scalar": ms_s.value, "mismatches": int(mism.value), "registers": int(regs.value)}

    def to_internal_order(self, ref_array: np.ndarray) -> np.ndarray:
        """Reorder a reference-order (n_states,) array into the engine's storage order."""
        perm = self.layout()["perm"]
        return np.ascontiguousarray(np.asarray(ref_array).reshape(tuple(self.grid_shape)).transpose(perm)).ravel()

    def expand_rows(self, action: int, s_begin: int = 0, count: int | None = None):
        """(idx, w, reward, terminated) in the reference's corner form, for parity checks."""
        self.build_table()
        lib = _ffi.lib()
        if count is None:
            count = self.n_states - s_begin
        Cn = 1 << self.N_DIMS
        idx = np.empty((count, Cn), dtype=np.int32)
        w = np.empty((count, Cn), dtype=np.float32)
        r = np.empty(count, dtype=np.float32)
        t = np.empty(count, dtype=np.uint8)
        _ffi.check(lib.pi_expand_rows(self._engine, int(action), int(s_begin), int(count), _ffi.ptr(idx), _ffi.ptr(w),
                                      _ffi.ptr(r), _ffi.ptr(t)))
        return idx, w, r, t


def _warm_start_source(source):
    """(values float32, bounds_low, bounds_high, grid_shape) of a warm-start source (see warm_start), validated on the
    host before any device work: a missing .npz entry raises KeyError, a dimensionality the C ABI cannot take raises
    ValueError, and a value count other than prod(grid_shape) raises EngineError (PI_ERR_INVALID)."""
    keys = ("value_function", "bounds_low", "bounds_high", "grid_shape")
    if isinstance(source, (str, Path)):
        path = Path(source).with_suffix(".npz")
        with np.load(path) as data:
            missing = [k for k in keys if k not in data.files]
            if missing:
                raise KeyError(f"{path}: warm-start source lacks {missing}")
            parts = [data[k] for k in keys]
    elif isinstance(source, tuple):
        if len(source) != 4:
            raise ValueError("a warm-start tuple is (values, bounds_low, bounds_high, grid_shape)")
        parts = list(source)
    else:
        parts = [getattr(source, k) for k in keys]
    values = np.ascontiguousarray(np.asarray(parts[0]).ravel(), dtype=np.float32)
    lo = np.asarray(parts[1], dtype=np.float32).ravel()
    hi = np.asarray(parts[2], dtype=np.float32).ravel()
    shape = np.asarray(parts[3], dtype=np.int64).ravel()
    if not 1 <= len(shape) <= _ffi.PI_MAX_DIMS or len(lo) != len(shape) or len(hi) != len(shape):
        raise ValueError(f"warm-start source: grid_shape {shape.tolist()} and bounds of {len(lo)} / {len(hi)} entries "
                         f"do not describe a 1..{_ffi.PI_MAX_DIMS}-D grid")
    if values.size != int(np.prod(shape)):
        raise _ffi.EngineError(_ffi.PI_ERR_INVALID, f"warm-start source has {values.size} values for a grid of shape "
                                                    f"{shape.tolist()} ({int(np.prod(shape))} states)")
    return values, lo, hi, shape


class CudaPolicyIteration2D(_CudaPolicyIterationBase):
    """Drop-in for the reference's CudaPolicyIteration2D (src/cuda_policy_iteration.py:46)."""
    N_DIMS = 2


class CudaPolicyIteration4D(_CudaPolicyIterationBase):
    """Drop-in for the reference's CudaPolicyIteration4D (src/cuda_policy_iteration.py:439)."""
    N_DIMS = 4


class CudaPolicyIteration6D(_CudaPolicyIterationBase):
    """Drop-in for the reference's CudaPolicyIteration6D (src/cuda_policy_iteration.py:847)."""
    N_DIMS = 6
