"""The plane-staged sweep's schedule and its stitched slot plan.

Every CTA of the sweep walks its chunks (c, c + grid, ... of the rotated schedule) as one sequence of steps: the loads of
a chunk's first step that the planner moved into slots the previous chunk no longer touches are issued one step ahead,
while that chunk's last step is still being backed up.  A wrong slot there corrupts V only under some timings, so these
tests replay every CTA's sequence on the host from the downloaded plan records and check the plan itself:
  * every (cell, outer corner) slot offset points at a slot that holds that corner's V-plane at that step;
  * no early load targets a slot the previous step of the same CTA reads or loads (chunk boundaries included);
  * no two loads of a step target one slot;
  * the schedule gives every CTA the same number of chunks and the same number of state-planes to within one;
and that the sweep run with that plan is bit-identical to the gather sweep."""
import numpy as np
import pytest

from dynamicprogramming_b200 import envs

pytestmark = pytest.mark.gpu

MAX_CELLS, MAX_OC, MAX_LOADS = 8, 16, 80
BAD_SLOT = 0xFFFF


def _prepared(env, bins, policy, monkeypatch):
    monkeypatch.setenv("DPB200_PLANE", "off")    # the engine's own sweeps stay on the gather kernels: they are the comparison
    eng = envs.make(env, bins=bins)
    eng.build_table()
    if policy == "greedy":
        eng.sweeps(3)
        eng.policy_improvement()
    else:   # many successor cells per state-plane: fallback cells, unstaged states
        eng.upload_policy(np.random.default_rng(7).integers(0, eng.n_actions, eng.n_states).astype(np.int32))
    eng.sweeps(5)
    return eng


def _decode(records):
    hdr = records[:, :4]
    cs = records[:, 16:16 + 2 * MAX_CELLS * MAX_OC].copy().view(np.uint16).reshape(-1, MAX_CELLS, MAX_OC)
    loads = records[:, 16 + 2 * MAX_CELLS * MAX_OC:].copy().view(np.uint32).reshape(-1, MAX_LOADS)
    return hdr[:, 0].astype(int), hdr[:, 1].astype(int), hdr[:, 2].astype(int), hdr[:, 3].astype(int), cs, loads


def _replay(out):
    """Walk every CTA's steps; returns the number of early loads at chunk starts that are not a CTA's first."""
    n_early, n_late, n_cells, flags, cs, loads = _decode(out["records"])
    begin, M, G, rot = out["chunk_begin"], out["n_chunks"], out["grid"], out["rot"]
    NS, noc, unit = out["slots"], out["noc"], out["pitch"] // 4
    assert M % G == 0 and begin[0] == 0 and begin[-1] == out["n_planes"] and np.all(np.diff(begin) > 0), (M, G)
    per_cta = [sum(int(begin[(ci + rot) % M + 1] - begin[(ci + rot) % M]) for ci in range(b, M, G)) for b in range(G)]
    assert max(per_cta) - min(per_cta) <= 1, (min(per_cta), max(per_cta))

    ooff = None   # V-plane offset of outer corner j from corner 0: the same for every cell of every plane
    stitched_early = 0
    for b in range(G):
        content = np.full(NS, -1, np.int64)   # V-plane each slot holds
        prev_touch = None                     # slots the previous step read or loaded
        for ci in range(b, M, G):
            c = (ci + rot) % M
            for pl in range(begin[c], begin[c + 1]):
                ne, nl = n_early[pl], n_late[pl]
                ld = loads[pl, :ne + nl]
                slots, vps = (ld >> 24).astype(int), (ld & 0xFFFFFF).astype(np.int64)
                assert np.all(slots < NS), pl
                assert len(set(slots.tolist())) == len(slots), f"plane {pl}: two loads into one slot"
                if prev_touch is not None:
                    bad = set(slots[:ne].tolist()) & prev_touch
                    assert not bad, f"plane {pl} (chunk {c}, CTA {b}): early loads into slots {bad} the previous step uses"
                    if pl == begin[c]:
                        stitched_early += ne
                content[slots] = vps
                K, fl = n_cells[pl], flags[pl]
                read = set()
                for k in range(K):
                    if (fl >> k) & 1:
                        assert np.all(cs[pl, k, :noc] == BAD_SLOT), pl
                        continue
                    s = cs[pl, k, :noc].astype(int) // unit
                    assert np.all(cs[pl, k, :noc] % unit == 0) and np.all(s < NS), pl
                    v = content[s]
                    assert np.all(v >= 0), f"plane {pl}: cell {k} reads a slot nothing was loaded into"
                    if ooff is None:
                        ooff = v - v[0]
                    assert np.array_equal(v - v[0], ooff), f"plane {pl}: cell {k} reads V-planes {v.tolist()}"
                    read |= set(s.tolist())
                prev_touch = read | set(slots.tolist())
    return stitched_early


CASES = [
    # (env, bins, cfg): default item mode; several chunks per CTA with short chunks; few slots (many late loads); one
    # state per thread (pack 0) with uneven chunks
    ("double_cartpole_swingup", 8, ""),
    ("double_cartpole_swingup", 8, "32,3,2,1,2"),
    ("double_cartpole_swingup", 10, ""),
    ("double_cartpole_swingup", 10, "0,0,2,2,0"),
    ("double_cartpole_swingup", 10, "36,7,1,2,0"),
    ("double_cartpole", 10, "0,5,2,1,2"),
]


@pytest.mark.parametrize("env,bins,cfg", CASES)
@pytest.mark.parametrize("policy", ["greedy", "random"])
@pytest.mark.parametrize("rot", [0, 37])
def test_stitched_plan_is_race_free_and_bit_identical(env, bins, cfg, policy, rot, monkeypatch):
    eng = _prepared(env, bins, policy, monkeypatch)
    out = eng.debug_plane_schedule(cfg, rot=rot, iters=2)
    assert out["rot"] == rot % out["n_chunks"]
    assert out["mismatches"] == 0, {k: v for k, v in out.items() if k not in ("records", "chunk_begin")}
    stitched = _replay(out)
    if policy == "greedy" and not cfg and out["n_chunks"] > out["grid"]:
        assert stitched > 0    # the chunk starts after a CTA's first do issue loads one step ahead
    eng.close()


def test_stitching_lowers_late_loads_on_a_k5_like_grid(monkeypatch):
    """At a chunk start the CTA's previous chunk still reads some slots: the rest take the first step's loads early."""
    eng = _prepared("double_cartpole_swingup", 10, "greedy", monkeypatch)
    out = eng.debug_plane_schedule("", rot=0, iters=1)
    n_early, n_late = _decode(out["records"])[:2]
    begin, M, G = out["chunk_begin"], out["n_chunks"], out["grid"]
    assert M > G, (M, G)
    starts = begin[G:M]   # chunk starts that are not a CTA's first (rotation 0)
    assert n_early[starts].sum() > 0.5 * (n_early[starts] + n_late[starts]).sum()
    np.testing.assert_allclose(out["late_per_plane"], n_late.sum() / out["n_planes"])
    eng.close()
