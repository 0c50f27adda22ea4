"""The engine at every dimensionality D = 1..6 against a plain host reference.

The shipped environments are 2-, 4- and 6-D, and the frozen parity hashes cover only those.  Odd D is the only case
with an odd number of row words (W = D + 2): the 4-byte row plane of the table builder, load_row / store_row and the
sweeps; D = 1 has no 16-byte plane and its own weight branch; D = 3 has 4-corner x-line windows; D = 5 runs the
plane-staged sweep with 8 outer corners.  The chain-of-integrators plugins of tests/fixtures/odd_dims.py use
explicitly rounded intrinsics only, so numpy float32 reproduces every row bit for bit, and everything the engine
computes from the rows is checked here against numpy:

* rows: index, weights, reward, terminated and absorbing, bit for bit, for every action;
* one sweep from adversarial V: a float64 backup within the bound of the fma chain, exact terminated / absorbing
  rows, the exact residual;
* every sweep family (persistent, JIT one-state and packed-pair, x-line, plane-staged) bit-identical to the
  ahead-of-time gather sweep, through the debug hooks and through a full run();
* improvement against float64 Q-values, exact tie-break and change count;
* run() against an exact sparse solve of the final policy's linear system;
* storage orders, host <-> device hand-off, save / load;
* lookup and closed-loop rollouts against numpy restatements.

The even dimensionalities run as controls: there the golden parity tests already pin the kernels, which shows that
the harness itself is right."""
import importlib.util
from pathlib import Path

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from dynamicprogramming_b200 import _ffi
from dynamicprogramming_b200.engine import CudaPIConfig

pytestmark = pytest.mark.gpu

_spec = importlib.util.spec_from_file_location("odd_dims", Path(__file__).resolve().parent / "fixtures" / "odd_dims.py")
odd = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(odd)

F32 = np.float32
U = 2.0 ** -24          # unit roundoff of float32
DIMS = [1, 2, 3, 4, 5, 6]
OFF = {"DPB200_PLANE": "off", "DPB200_XLINE": "off", "DPB200_PAIR": "off", "DPB200_PERSIST": "off"}


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def _engine(D, monkeypatch, config=None, **env):
    """A fixture engine; the JIT sweeps stay off unless `env` turns one on, so the engine's own sweeps are the
    ahead-of-time gather sweep (pi::eval_sweep_kernel<D>)."""
    monkeypatch.delenv("DPB200_FAST_DIM", raising=False)
    for k, v in {**OFF, **env}.items():
        monkeypatch.setenv(k, v)
    return odd.make(D, config)


# ── host reference ─────────────────────────────────────────────────────────────────────────────────────────────────

def _corner_bit(D, c, d):
    """Corner enumeration of the reference's rows: at D = 2 dim 0 is the high bit, otherwise bit d is dim d."""
    return (c >> (1 - d)) & 1 if D == 2 else (c >> d) & 1


def host_rows(eng, a):
    """The table builder's row of every state for action `a` in expand_rows form, from numpy float32: the step, then
    get_barycentric_Nd's cell search n = (x - lo) / (hi - lo) * (shape - 1), clamp, i = min(trunc(n), shape - 2),
    f = n - i, and corner weights as prefix products in dimension order.  code: 0 live, 1 terminated, 2 absorbing."""
    D, N = eng.N_DIMS, eng.n_states
    C = 1 << D
    states = eng.states_space
    shape = [int(s) for s in eng.grid_shape]
    stride = np.array(eng.strides, np.int64)
    nx, r, term = odd.step_numpy(states, odd.ACTIONS[a])
    absorbing = odd.terminal_mask(states)
    code = np.where(absorbing, 2, np.where(term, 1, 0)).astype(np.uint8)
    live = code == 0
    idx = np.where(code == 1, -1, -2).astype(np.int64)[:, None].repeat(C, axis=1)
    w = np.zeros((N, C), F32)
    base = np.zeros(int(live.sum()), np.int64)
    fr = np.empty((int(live.sum()), D), F32)
    for d in range(D):
        lo, hi = F32(eng.bounds_low[d]), F32(eng.bounds_high[d])
        pn = ((nx[live, d] - lo).astype(F32) / F32(hi - lo)).astype(F32)
        pn = (pn * F32(shape[d] - 1)).astype(F32)
        pn = np.maximum(F32(0), np.minimum(pn, F32(shape[d] - 1)))
        i = np.minimum(pn.astype(np.int64), shape[d] - 2)
        base += i * stride[d]
        fr[:, d] = (pn - i.astype(F32)).astype(F32)
    for c in range(C):
        off = sum(_corner_bit(D, c, d) * int(stride[d]) for d in range(D))
        idx[live, c] = base + off
        wc = np.ones(len(base), F32)
        for d in range(D):
            wc = (wc * (fr[:, d] if _corner_bit(D, c, d) else (F32(1) - fr[:, d]).astype(F32))).astype(F32)
        w[live, c] = wc
    return idx, w, np.where(absorbing, F32(0), r).astype(F32), code


def all_host_rows(eng):
    rows = [host_rows(eng, a) for a in range(eng.n_actions)]
    return tuple(np.stack([r[k] for r in rows]) for k in range(4))   # (A, N, C) idx / w, (A, N) reward / code


def q_values(rows, V, gamma):
    """float64 backups of every (action, state) from the rows and V: r + gamma * sum_c w_c V_c (live), r (terminated),
    V (absorbing); and the bound of the float32 fma chain that computes them on the device,
    (C + 2) u (gamma sum_c |w_c V_c| + |r|) with C = 2^D corners."""
    idx, w, r, code = rows
    C = idx.shape[2]
    g = float(F32(gamma))
    Vd = V.astype(np.float64)
    wv = w.astype(np.float64) * Vd[np.maximum(idx, 0)]
    wv[code != 0] = 0.0
    q = r.astype(np.float64) + g * wv.sum(axis=2)
    q = np.where(code == 2, Vd[None, :], q)
    tol = (C + 2) * U * (g * np.abs(wv).sum(axis=2) + np.abs(r.astype(np.float64)))
    return q, tol


def _set_policy(eng, policy, seed=7):
    if policy == "greedy":
        eng.sweeps(3)
        eng.policy_improvement()
    elif policy == "random":
        eng.upload_policy(np.random.default_rng(seed).integers(0, eng.n_actions, eng.n_states).astype(np.int32))


# ── 1. rows ────────────────────────────────────────────────────────────────────────────────────────────────────────

@pytest.mark.parametrize("D", DIMS)
def test_rows_equal_the_host_step_and_cell_search(D, monkeypatch):
    eng = _engine(D, monkeypatch)
    eng.build_table()
    kinds = np.zeros(3, np.int64)
    clamped = [np.zeros(2, bool) for _ in range(D)]
    for a in range(eng.n_actions):
        idx, w, r, t = eng.expand_rows(a)
        hidx, hw, hr, hcode = host_rows(eng, a)
        np.testing.assert_array_equal(t, hcode, err_msg=f"D={D} action {a}: terminated / absorbing")
        np.testing.assert_array_equal(idx, hidx, err_msg=f"D={D} action {a}: corner index")
        np.testing.assert_array_equal(bits(w), bits(hw), err_msg=f"D={D} action {a}: corner weight")
        np.testing.assert_array_equal(bits(r), bits(hr), err_msg=f"D={D} action {a}: reward")
        kinds += np.bincount(t, minlength=3)
        nx, _, _ = odd.step_numpy(eng.states_space, odd.ACTIONS[a])
        for d in range(D):
            clamped[d] |= [(nx[t == 0, d] < eng.bounds_low[d]).any(), (nx[t == 0, d] > eng.bounds_high[d]).any()]
    # the fixture reaches every kind of row: live, terminated, absorbing, and clamps on both sides of every dimension
    assert (kinds > 0).all(), kinds
    assert all(c.all() for c in clamped), clamped
    # the duplicated action has bit-equal rows
    a, b = odd.TIED_ACTIONS
    for x, y in zip(eng.expand_rows(a), eng.expand_rows(b)):
        np.testing.assert_array_equal(np.ascontiguousarray(x).view(np.uint8), np.ascontiguousarray(y).view(np.uint8))
    eng.close()


# ── 2. one sweep from adversarial values ───────────────────────────────────────────────────────────────────────────

def _adversarial_values(N, seed):
    rng = np.random.default_rng(seed)
    V = (rng.choice([-1.0, 1.0], N) * 10.0 ** rng.uniform(-12, 12, N)).astype(F32)
    V[rng.random(N) < 0.05] = F32(0.0)
    V[rng.random(N) < 0.05] = F32(-0.0)
    return V


@pytest.mark.parametrize("D", DIMS)
def test_one_sweep_from_adversarial_values_matches_a_float64_backup(D, monkeypatch):
    eng = _engine(D, monkeypatch)
    eng.build_table()
    N = eng.n_states
    rng = np.random.default_rng(100 + D)
    V0 = _adversarial_values(N, D)
    P = rng.integers(0, eng.n_actions, N).astype(np.int32)
    eng.upload_values(V0)
    eng.upload_policy(P)
    res, _ = eng.sweeps(1)
    v1, p1 = eng.download()
    np.testing.assert_array_equal(p1, P)
    rows = all_host_rows(eng)
    q, tol = q_values(rows, V0, eng.config.gamma)
    s = np.arange(N)
    q, tol, code, r = q[P, s], tol[P, s], rows[3][P, s], rows[2][P, s]
    live = code == 0
    err = np.abs(v1[live].astype(np.float64) - q[live])
    assert (err <= tol[live]).all(), (D, float((err / np.maximum(tol[live], 1e-300)).max()))
    np.testing.assert_array_equal(v1[code == 1], r[code == 1])                  # terminated: exactly r
    np.testing.assert_array_equal(bits(v1[code == 2]), bits(V0[code == 2]))     # absorbing: V itself, bit for bit
    assert (code == 1).any() and (code == 2).any()
    assert F32(res) == np.abs(v1 - V0).max()                                   # the residual, exactly
    eng.close()


# ── 3. every sweep family is bit-identical to the gather sweep ─────────────────────────────────────────────────────

def _xline_cfgs(eng):
    """x-line configurations (K = 2 and 4, roll 1 and 2) with the tile filled from the fastest non-fast position."""
    D, perm = eng.N_DIMS, eng.layout()["perm"]
    S = int(eng.grid_shape[0])
    out = []
    for cfg in ("2,0,4,8,2,1", "4,0,4,8,1,1", "4,0,2,4,1,2"):
        K, warps = int(cfg.split(",")[0]), int(cfg.split(",")[3])
        slots, tile = warps * (32 // (S // K)), [1] * (D - 1)
        for k in range(D - 2, -1, -1):
            n = int(eng.grid_shape[perm[k]])
            tile[k] = max(t for t in range(1, n + 1) if n % t == 0 and t <= slots)
            slots //= tile[k]
        out.append(cfg + ":" + ",".join(map(str, tile)))
    return out


PAIR_CFGS = [(64, 8, 1, 0, 0), (128, 8, 2, 8, 1), (256, 2, 1, 0, 1)]   # threads, minb, lv, group, single
PLANE_CFGS = ["0,0,2,2,2", "0,0,2,2,0", "0,3,1,1,1"]                  # item mode, one state per thread, few slots


def _layout_env(D):
    return "0,1" if D >= 4 else "0"       # the x-line sweep needs dim 0 fastest, the plane sweep (dim 0, dim 1)


@pytest.mark.parametrize("D", DIMS)
@pytest.mark.parametrize("policy", ["initial", "greedy", "random"])
def test_jit_sweeps_are_bit_identical_to_the_gather_sweep(D, policy, monkeypatch):
    eng = _engine(D, monkeypatch, DPB200_FAST_DIM=_layout_env(D))
    eng.build_table()
    assert eng.eval_kernel_info()["kernel"] == f"pi::eval_sweep_kernel<{D}>"
    _set_policy(eng, policy)
    eng.sweeps(4)
    for cfg in PAIR_CFGS:
        if D < 3:
            with pytest.raises(_ffi.EngineError, match="needs D >= 3"):
                eng.debug_pair(*cfg[:2], iters=1, lv=cfg[2], group=cfg[3], single=cfg[4])
            continue
        out = eng.debug_pair(*cfg[:2], iters=1, lv=cfg[2], group=cfg[3], single=cfg[4])
        assert out["mismatches"] == 0, (cfg, out)
    if D < 3:
        with pytest.raises(_ffi.EngineError, match="needs 3 <= D <= 6"):
            eng.debug_xline("2,0,4,8,2,1:" + ",".join(["1"] * max(D - 1, 1)), iters=1)
    else:
        windows = []
        for cfg in _xline_cfgs(eng):
            out = eng.debug_xline(cfg, iters=1)
            assert out["mismatches"] == 0, (cfg, out)
            windows.append(out["window_fraction"])
        if policy != "random":
            assert max(windows) > 0, windows                      # the vector-window path is taken
    if D < 4:
        with pytest.raises(_ffi.EngineError, match="needs 4 <= D <= 6"):
            eng.debug_plane("", iters=1)
    else:
        assert eng.layout()["fast_dim2"] == 1
        for cfg in PLANE_CFGS:
            out = eng.debug_plane(cfg, iters=1)
            assert out["mismatches"] == 0, (cfg, out)
    eng.close()


_RUNS: dict = {}


def _result(eng):
    return eng.pi_iterations, eng.total_eval_sweeps, eng.policy.copy(), bits(eng.value_function).copy()


def _gather_run(D, monkeypatch):
    """run() on the ahead-of-time gather sweep in the reference storage order (computed once per D)."""
    if D not in _RUNS:
        eng = _engine(D, monkeypatch, DPB200_FAST_DIM="ref")
        eng.build_table()
        assert eng.eval_kernel_info()["kernel"] == f"pi::eval_sweep_kernel<{D}>"
        eng.run()
        assert eng.converged
        _RUNS[D] = _result(eng)
    return _RUNS[D]


def _assert_same_run(got, want, what):
    assert got[:2] == want[:2], what
    np.testing.assert_array_equal(got[2], want[2], err_msg=f"{what}: policy")
    np.testing.assert_array_equal(got[3], want[3], err_msg=f"{what}: value function bits")


FAMILIES = {
    # name: (environment, the kernel eval_kernel_info() names, smallest D, largest D)
    "persistent": ({"DPB200_PERSIST": "on"}, "eval_persistent_kernel", 1, 4),
    "gp_pair": ({"DPB200_PAIR": "force:64,8"}, "gp_sweep (packed pairs", 3, 6),
    "gp_single": ({"DPB200_PAIR": "force:128,8,2,8,1"}, "gp_sweep (one state/thread", 3, 6),
    "xline": ({"DPB200_XLINE": "force:2,0,4,8,2,1:" + ",".join(["1"] * 5), "DPB200_FAST_DIM": "0"}, "xl_sweep", 3, 6),
    "plane_items": ({"DPB200_PLANE": "force:0,0,2,2,2"}, "ps_sweep", 4, 6),
    "plane_single": ({"DPB200_PLANE": "force:0,0,2,2,0"}, "ps_sweep", 4, 6),
}


@pytest.mark.parametrize("D", DIMS)
@pytest.mark.parametrize("family", list(FAMILIES))
def test_full_run_with_each_sweep_family_forced_equals_the_gather_sweep(D, family, monkeypatch):
    """Where a family cannot take D: the persistent sweep is eligible for D <= 4 only and the JIT one-state /
    packed-pair and x-line sweeps need D >= 3 (pair_prepare, xline_applicable); the engine then keeps the gather
    sweep.  DPB200_PLANE=force fails at D < 4 (plane_applicable)."""
    want = _gather_run(D, monkeypatch)
    env, name, d_min, d_max = FAMILIES[family]
    env = {"DPB200_FAST_DIM": _layout_env(D), **env}
    eng = _engine(D, monkeypatch, **env)
    if family.startswith("plane") and D < 4:
        with pytest.raises(_ffi.EngineError, match="DPB200_PLANE=force: needs 4 <= D <= 6"):
            eng.build_table()
        eng.close()
        return
    eng.build_table()
    kernel = eng.eval_kernel_info()["kernel"]
    if d_min <= D <= d_max:
        assert name in kernel, kernel
    else:
        assert kernel == f"pi::eval_sweep_kernel<{D}>", kernel
    eng.run()
    _assert_same_run(_result(eng), want, f"D={D} {family}")


# ── 4. improvement ─────────────────────────────────────────────────────────────────────────────────────────────────

@pytest.mark.parametrize("D", DIMS)
def test_improvement_matches_float64_q_values(D, monkeypatch):
    eng = _engine(D, monkeypatch)
    eng.build_table()
    N = eng.n_states
    rows = all_host_rows(eng)
    code = rows[3][0]
    s = np.arange(N)
    rng = np.random.default_rng(200 + D)
    eng.sweeps(40)
    smooth, _ = eng.download()
    for V in (_adversarial_values(N, 300 + D), smooth):
        P0 = rng.integers(0, eng.n_actions, N).astype(np.int32)
        eng.upload_values(V)
        eng.upload_policy(P0)
        stable = eng.policy_improvement()
        _, P1 = eng.download()
        q, tol = q_values(rows, V, eng.config.gamma)
        best = q.argmax(axis=0)
        live = code != 2
        gap = q[best, s] - q[P1, s]
        assert (gap[live] <= (tol[best, s] + tol[P1, s])[live]).all(), float(gap[live].max())
        assert not (P1[live] == odd.TIED_ACTIONS[1]).any()            # bit-equal rows: the lower index wins
        assert (P1[live] == odd.TIED_ACTIONS[0]).any()
        np.testing.assert_array_equal(P1[~live], P0[~live])           # absorbing states keep their action
        assert eng.last_changed == int((P1 != P0).sum())
        assert stable == (eng.last_changed == 0)
    eng.close()


# ── 5. run() against an exact solve ────────────────────────────────────────────────────────────────────────────────

@pytest.mark.parametrize("D", DIMS)
def test_run_matches_an_exact_solve_of_its_policy(D, monkeypatch):
    """Evaluation stops after a sweep whose residual is below theta.  For that sweep V' = T~V = TV + e with
    |e| <= eps (the fma-chain bound), so (1 - gamma) |V' - V_pi| <= gamma |V' - V| + eps < gamma theta + eps."""
    cfg = CudaPIConfig(gamma=odd.GAMMA, theta=1e-5, max_eval_iter=10_000, max_pi_iter=50)
    eng = _engine(D, monkeypatch, config=cfg)
    eng.build_table()
    rows = all_host_rows(eng)
    eng.run()
    assert eng.converged
    V, P = eng.value_function, eng.policy
    N = eng.n_states
    s = np.arange(N)
    idx, w, r, code = (x[P, s] for x in rows)
    g = float(F32(cfg.gamma))
    live = code == 0
    C = idx.shape[1]
    rr = np.repeat(s[live], C)
    A = sp.identity(N, format="csr") - sp.csr_matrix((g * w[live].astype(np.float64).ravel(), (rr, idx[live].ravel())),
                                                     shape=(N, N))
    b = np.where(code == 2, odd.TERMINAL_VALUE, r.astype(np.float64))
    v_pi = spla.spsolve(A.tocsc(), b)
    q, tol = q_values(rows, V, cfg.gamma)
    eps = 1.01 * tol[P, s].max()
    theta = float(F32(cfg.theta)) * (1 + 2.0 ** -22)
    bound = (g * theta + eps) / (1 - g)
    err = np.abs(V.astype(np.float64) - v_pi)
    assert err.max() <= bound, (float(err.max()), bound)
    np.testing.assert_array_equal(V[code == 2], F32(odd.TERMINAL_VALUE))
    # the policy is greedy with respect to its own V
    best = q.argmax(axis=0)
    gap = q[best, s] - q[P, s]
    assert (gap <= tol[best, s] + tol[P, s]).all(), float(gap.max())


# ── 6. storage order and hand-off ──────────────────────────────────────────────────────────────────────────────────

@pytest.mark.parametrize("D", DIMS)
def test_storage_order_never_changes_results(D, monkeypatch):
    want = _gather_run(D, monkeypatch)
    for fast in ["0", "auto"] + (["0,1"] if D >= 4 else []):
        eng = _engine(D, monkeypatch, DPB200_FAST_DIM=fast)
        lay = eng.layout()
        if fast != "auto":
            assert lay["fast_dim"] == 0
        if fast == "0,1":
            assert lay["perm"][-2:] == [1, 0], lay
        eng.run()
        _assert_same_run(_result(eng), want, f"D={D} DPB200_FAST_DIM={fast}")


@pytest.mark.parametrize("D", DIMS)
def test_host_device_handoff_and_save_load(D, monkeypatch, tmp_path):
    eng = _engine(D, monkeypatch, DPB200_FAST_DIM="0")
    eng.build_table()
    N = eng.n_states
    rng = np.random.default_rng(400 + D)
    V = rng.standard_normal(N).astype(F32)
    P = rng.integers(0, eng.n_actions, N).astype(np.int32)
    eng.upload_values(V)
    eng.upload_policy(P)
    v2, p2 = eng.download()
    np.testing.assert_array_equal(bits(v2), bits(V))
    np.testing.assert_array_equal(p2, P)
    lay = eng.layout()
    assert lay["perm"][-1] == 0 and sorted(lay["perm"]) == list(range(D))
    internal = eng.to_internal_order(V)
    expect = V.reshape(tuple(eng.grid_shape)).transpose(lay["perm"]).ravel()
    np.testing.assert_array_equal(bits(internal), bits(expect))
    np.testing.assert_array_equal(bits(eng.d_value_function.raw()), bits(internal))
    np.testing.assert_array_equal(eng.d_policy.raw(), eng.to_internal_order(P))
    np.testing.assert_array_equal(eng.d_policy.get(), P)
    eng.sweeps(3)
    v_full, _ = eng.download()
    eng.close()
    # the storage-order slice upload gives the same sweeps as the reference-order upload
    eng = _engine(D, monkeypatch, DPB200_FAST_DIM="0")
    eng.build_table()
    eng.upload_values(V)
    eng.upload_policy_local(eng.to_internal_order(P))
    eng.sweeps(3)
    v_local, p_local = eng.download()
    np.testing.assert_array_equal(bits(v_local), bits(v_full))
    np.testing.assert_array_equal(p_local, P)
    eng.run()
    eng.save(tmp_path / "p")
    d = np.load(tmp_path / "p.npz")
    assert list(d.files) == ["value_function", "policy", "bounds_low", "bounds_high", "grid_shape", "strides",
                             "corner_bits", "action_space", "states_space"]
    assert d["corner_bits"].shape == (1 << D, D)
    np.testing.assert_array_equal(d["corner_bits"][:, ::-1], (np.arange(1 << D)[:, None] >> np.arange(D)) & 1)
    assert d["states_space"].shape == (N, D)
    np.testing.assert_array_equal(d["grid_shape"], odd.SHAPES[D])
    loaded = odd.plugin_class(D).load(tmp_path / "p.npz")
    np.testing.assert_array_equal(loaded.policy, eng.policy)
    np.testing.assert_array_equal(bits(loaded.value_function), bits(eng.value_function))
    np.testing.assert_array_equal(bits(loaded.states_space), bits(eng.states_space))


# ── 7. lookup and rollout ──────────────────────────────────────────────────────────────────────────────────────────

def lookup_numpy(policy, actions, lo, hi, shape, pts):
    """lookup_point (csrc/lookup_src.cuh) restated in numpy: float64 t and weight products, corner_bits order (dim 0
    the most significant bit), float32 ascending sum."""
    pts = np.asarray(pts, F32)
    n, D = pts.shape
    shape = [int(s) for s in shape]
    stride = [int(np.prod(shape[d + 1:])) for d in range(D)]
    base = np.empty((n, D), np.int64)
    t = np.empty((n, D), np.float64)
    for d in range(D):
        l, h = F32(lo[d]), F32(hi[d])
        step = F32(np.float64(F32(h - l)) / np.float64(shape[d] - 1))
        q = np.where(pts[:, d] < h, pts[:, d], h)
        q = np.where(q > l, q, l).astype(F32)
        cell = ((q - l).astype(F32) / step).astype(F32)
        i = cell.astype(np.int64)
        i = np.where(i >= shape[d] - 1, shape[d] - 2, i)
        base[:, d] = i
        num = q.astype(np.float64) - (np.float64(l) + i.astype(np.float64) * np.float64(step))
        t[:, d] = (num / np.float64(step)).astype(F32).astype(np.float64)
    acc = np.zeros(n, F32)
    act = np.asarray(actions, F32)
    for c in range(1 << D):
        w = np.ones(n, np.float64)
        flat = np.zeros(n, np.int64)
        for d in range(D):
            bit = (c >> (D - 1 - d)) & 1
            w = w * (t[:, d] if bit else 1.0 - t[:, d])
            flat += (base[:, d] + bit) * stride[d]
        acc = (acc + (w.astype(F32) * act[policy[flat]]).astype(F32)).astype(F32)
    return acc


def lookup_exact(policy, actions, lo, hi, shape, pts):
    """Multilinear interpolation in float64 on the uniform grid lo + i (hi - lo) / (shape - 1), queries clamped."""
    pts = np.asarray(pts, np.float64)
    n, D = pts.shape
    shape = [int(s) for s in shape]
    stride = [int(np.prod(shape[d + 1:])) for d in range(D)]
    base = np.empty((n, D), np.int64)
    t = np.empty((n, D))
    for d in range(D):
        l, h = float(lo[d]), float(hi[d])
        x = (np.clip(pts[:, d], l, h) - l) / (h - l) * (shape[d] - 1)
        base[:, d] = np.minimum(np.floor(x).astype(np.int64), shape[d] - 2)
        t[:, d] = x - base[:, d]
    out = np.zeros(n)
    for c in range(1 << D):
        w = np.ones(n)
        flat = np.zeros(n, np.int64)
        for d in range(D):
            bit = (c >> (D - 1 - d)) & 1
            w *= t[:, d] if bit else 1.0 - t[:, d]
            flat += (base[:, d] + bit) * stride[d]
        out += w * np.asarray(actions, np.float64)[policy[flat]]
    return out


def query_points(eng, seed):
    """Every grid node, and random points whose coordinates are, per dimension, a node, a node +/- 1 ulp, lo, hi,
    hi - 1 ulp, outside on either side, +/- inf or uniform over a widened box."""
    rng = np.random.default_rng(seed)
    D = eng.N_DIMS
    lo, hi = eng.bounds_low.astype(F32), eng.bounds_high.astype(F32)
    n = 4000
    pts = (lo + (hi - lo) * rng.uniform(-0.2, 1.2, (n, D))).astype(F32)
    axes = [np.linspace(*odd.RANGES[d], int(eng.grid_shape[d]), dtype=F32) for d in range(D)]
    for d in range(D):
        kind = rng.integers(0, 10, n)
        node = axes[d][rng.integers(0, len(axes[d]), n)]
        special = [node, np.nextafter(node, F32(np.inf)), np.nextafter(node, F32(-np.inf)), np.full(n, lo[d]),
                   np.full(n, hi[d]), np.full(n, np.nextafter(hi[d], F32(-np.inf))),
                   np.full(n, lo[d] - F32(0.5)), np.full(n, hi[d] + F32(0.5)), np.full(n, F32(np.inf)),
                   np.full(n, F32(-np.inf))]
        for k in range(10):
            m = (kind == k) & (rng.random(n) < 0.6)
            pts[m, d] = special[k][m]
    return np.concatenate([eng.states_space, pts]).astype(F32)


@pytest.mark.parametrize("D", DIMS)
def test_lookup_matches_numpy_restatements(D, monkeypatch, tmp_path):
    eng = _engine(D, monkeypatch, DPB200_FAST_DIM="0")
    eng.build_table()
    eng.sweeps(10)
    eng.policy_improvement()
    _, pol = eng.download()
    pts = query_points(eng, 500 + D)
    args = (eng.action_space, eng.bounds_low, eng.bounds_high, eng.grid_shape, pts)
    live = eng.lookup_actions(pts)                  # the device-resident policy, in the engine's storage order
    np.testing.assert_array_equal(bits(live), bits(lookup_numpy(pol, *args)))
    np.testing.assert_allclose(live, lookup_exact(pol, *args), rtol=0, atol=1e-4)
    eng.run()
    eng.save(tmp_path / "p")
    loaded = odd.plugin_class(D).load(tmp_path / "p.npz")
    got = loaded.lookup_actions(pts)                 # PolicyLookup over the saved reference-order policy
    np.testing.assert_array_equal(bits(got), bits(lookup_numpy(loaded.policy, *args)))
    np.testing.assert_allclose(got, lookup_exact(loaded.policy, *args), rtol=0, atol=1e-4)


def rollout_numpy(policy, eng, x0, T, gamma):
    """Closed-loop episodes as a numpy loop: lookup_numpy + odd.step_numpy; returns in float64 (total += r,
    ret += disc * r, disc *= gamma); NaN after each episode's end."""
    n, D = x0.shape
    S = np.full((n, T + 1, D), np.nan, F32)
    A = np.full((n, T), np.nan, F32)
    R = np.full((n, T), np.nan, F32)
    S[:, 0] = x0
    x = x0.copy()
    length = np.zeros(n, np.int32)
    term = np.zeros(n, bool)
    total, ret, disc = np.zeros(n), np.zeros(n), np.ones(n)
    for t in range(T):
        alive = np.nonzero(~term)[0]
        if len(alive) == 0:
            break
        a = lookup_numpy(policy, eng.action_space, eng.bounds_low, eng.bounds_high, eng.grid_shape, x[alive])
        nx, r, tm = odd.step_numpy(x[alive], a)
        A[alive, t], R[alive, t], S[alive, t + 1] = a, r, nx
        x[alive] = nx
        length[alive] = t + 1
        term[alive] = tm
        rd = r.astype(np.float64)
        total[alive] = total[alive] + rd
        ret[alive] = ret[alive] + disc[alive] * rd
        disc[alive] = disc[alive] * np.float64(gamma)
    return dict(states=S, actions=A, rewards=R, length=length, terminated=term, final_states=x, total_reward=total,
                discounted_return=ret)


@pytest.mark.parametrize("D", DIMS)
def test_rollout_matches_a_numpy_loop(D, monkeypatch):
    eng = _engine(D, monkeypatch)
    eng.build_table()
    N = eng.n_states
    rng = np.random.default_rng(600 + D)
    # full push right on the right of dim 0 (episodes terminate), full push left on the left (episodes leave the grid and
    # run out), random actions in between
    x = eng.states_space[:, 0]
    P = np.where(x > 0.3, 4, np.where(x < -0.3, 0, rng.integers(0, eng.n_actions, N))).astype(np.int32)
    eng.upload_policy(P)
    lo, hi = eng.bounds_low, eng.bounds_high
    x0 = (lo + (hi - lo) * rng.uniform(-0.1, 1.1, (500, D))).astype(F32)
    T = 40
    gamma = float(F32(odd.GAMMA))
    got = eng.rollout(x0, T, record=True)
    exp = rollout_numpy(P, eng, x0, T, gamma)
    np.testing.assert_array_equal(got.length, exp["length"])
    np.testing.assert_array_equal(got.terminated, exp["terminated"])
    for name in ("states", "actions", "rewards", "final_states", "total_reward", "discounted_return"):
        np.testing.assert_array_equal(bits(getattr(got, name)), bits(exp[name]), err_msg=f"D={D} {name}")
    assert got.terminated.any() and (got.length == T).any()
    eng.close()
