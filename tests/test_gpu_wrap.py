"""GPU parity of wrap-around trees (ghost identities, ghostPoint.jl:60-111) and of the two-pass range kernel.

Every wrap configuration of tests/wrap_model.py (one to four wrap dimensions, wraps on the grid axes x, y, z and
off them), with points and queries on the seams, at radii on both sides of the period / 2 bound of the ghost-pair
path and beyond the period.  Range results: index sets equal, no duplicates, keys equal as bit patterns, against
the CPU oracle for the whole batch and against the brute-force model (which test_wrap_model.py pins to the oracle)
for a sample.  Nearest: node and distance bits.  Also: the two-pass kernel forced on unwrapped trees, and the
consumers of wrapped trees that must refuse or notice what they cannot serve."""
import math
import os

import numpy as np
import pytest

import oracle
import wrap_model as M
from rrtqx_3d_b200 import _abi as A
from rrtqx_3d_b200 import workloads as W
from rrtqx_3d_b200.device import DeviceTree, EdgeSet, PolygonSet, SphereSet, extend_query

pytestmark = pytest.mark.gpu

N_POINTS = 2000
CONFIG_NAMES = list(M.CONFIGS)


def _canon(counts, offsets, idx, dist):
    """CSR result (lists in any order and place) -> (counts, idx, dist) with each query's list in ascending node
    order, queries in order.  Fails on a duplicate within a list."""
    counts = np.asarray(counts, dtype=np.int64)
    nq = len(counts)
    start = np.asarray(offsets[:nq], dtype=np.int64)
    q_of = np.repeat(np.arange(nq, dtype=np.int64), counts)
    first = np.repeat(np.cumsum(counts) - counts, counts)
    pos = np.repeat(start, counts) + (np.arange(len(q_of), dtype=np.int64) - first)
    gi = idx[pos].astype(np.int64)
    order = np.argsort(q_of * (1 << 32) + gi, kind="stable")
    gi, q_sorted = gi[order], q_of[order]
    dup = (gi[1:] == gi[:-1]) & (q_sorted[1:] == q_sorted[:-1])
    assert not dup.any(), f"duplicate node {gi[1:][dup][0]} in the list of query {q_sorted[1:][dup][0]}"
    return counts, gi, (dist[pos][order] if dist is not None else None)


def _gpu(t, qs, r, ranges=None, want_dist=True):
    res, total = t.range_query(qs, r if ranges is None else 0.0, ranges=ranges, want_dist=want_dist)
    counts, offsets = res.layout()
    idx, dist = res.fetch(want_dist)
    assert total == counts.sum()
    return _canon(counts, offsets, idx, dist)


def _orc(orc, qs, r=None, ranges=None):
    if ranges is None:
        counts, offsets, idx, key = orc.range_batch(r, qs, nthreads=8)
        return _canon(counts, offsets, idx, key)
    lists = []
    for q, rr in zip(qs, ranges):
        oi, ok = orc.find_within_range(rr, q)
        orc.empty(oi)
        lists.append((oi, ok))
    counts = np.array([len(i) for i, _ in lists], dtype=np.int64)
    offsets = np.concatenate([[0], np.cumsum(counts)])
    idx = np.concatenate([i for i, _ in lists]) if counts.sum() else np.zeros(0, np.int32)
    key = np.concatenate([k for _, k in lists]) if counts.sum() else np.zeros(0)
    return _canon(counts, offsets, idx, key)


def _same(a, b, what):
    assert np.array_equal(a[0], b[0]), f"{what}: counts differ (first query {np.nonzero(a[0] != b[0])[0][:1]})"
    assert np.array_equal(a[1], b[1]), f"{what}: index sets differ"
    if a[2] is not None and b[2] is not None:
        assert np.array_equal(a[2].view(np.uint64), b[2].view(np.uint64)), f"{what}: keys differ"


def _sample(nq):
    """The edge placements in front of every query set, then a stride sample."""
    return sorted(set(range(min(nq, 64))) | set(range(64, nq, 97)))


def _model(pts, qs, r, cfg, got, ranges=None):
    _, wraps, wps, _ = cfg
    off = np.concatenate([[0], np.cumsum(got[0])])
    for qi in _sample(len(qs)):
        rr = r if ranges is None else ranges[qi]
        mi, mk = M.range_query(pts, qs[qi], rr, wraps, wps)
        gi, gk = got[1][off[qi]:off[qi + 1]], got[2][off[qi]:off[qi + 1]]
        assert np.array_equal(gi, mi), f"query {qi}, r = {rr!r}: index set differs from the model"
        assert np.array_equal(gk.view(np.uint64), mk.view(np.uint64)), f"query {qi}, r = {rr!r}: keys differ from the model"


class _TwoPass:
    """RRTQX_RANGE_TWO_PASS for the duration of a with-block (the switch is read at context creation and reload)."""

    def __init__(self, ctx):
        self.ctx = ctx

    def __enter__(self):
        os.environ["RRTQX_RANGE_TWO_PASS"] = "1"
        self.ctx.reload_tuning()

    def __exit__(self, *exc):
        del os.environ["RRTQX_RANGE_TWO_PASS"]
        self.ctx.reload_tuning()


def _trees(ctx, cfg, n=N_POINTS):
    d, wraps, wps, _ = cfg
    pts = M.points(1, n, cfg)
    orc = oracle.KDTree(d, wraps, wps)
    orc.insert_batch(pts)
    t = DeviceTree(ctx, d, wraps=wraps, wrap_points=wps)
    t.insert_batch(pts)
    return pts, orc, t


@pytest.mark.parametrize("name", CONFIG_NAMES)
def test_wrapped_range_every_radius_and_path(ctx, name):
    """2049 queries (sorted-query path) at every radius through the path the library picks, and through the
    two-pass kernel where that is a different path; count-only and no-dist calls agree with the full call."""
    cfg = M.CONFIGS[name]
    d, wraps, wps, _ = cfg
    pts, orc, t = _trees(ctx, cfg)
    qs = M.queries(2, 2049, cfg, pts)
    for r in M.radii(wps):
        got = _gpu(t, qs, r)
        _same(got, _orc(orc, qs, r), f"{name} r = {r!r}")
        _model(pts, qs, r, cfg, got)
        if len(wraps) == 1 and r <= 0.5 * wps[0]:     # the ghost-pair path ran: the two-pass kernel must agree
            with _TwoPass(ctx):
                _same(_gpu(t, qs, r), got, f"{name} r = {r!r}, two-pass vs ghost pairs")
        res, total = t.range_query(qs, r, want_dist=False, count_only=True)
        assert total == got[0].sum() and np.array_equal(res.layout()[0], got[0])
        nodist = _gpu(t, qs, r, want_dist=False)
        assert np.array_equal(nodist[0], got[0]) and np.array_equal(nodist[1], got[1])


@pytest.mark.parametrize("name", CONFIG_NAMES)
def test_wrapped_range_batch_sizes_and_unsorted_tail(ctx, name):
    """Batches of 1, 3 and 5000 queries, then a tail of single inserts (on the seams too) and the queries again."""
    cfg = M.CONFIGS[name]
    d, wraps, wps, _ = cfg
    pts, orc, t = _trees(ctx, cfg)
    qs = M.queries(3, 5000, cfg, pts)
    rs = M.radii(wps)
    for nq in (1, 3):
        for r in rs:
            sub = np.ascontiguousarray(qs[:nq])
            got = _gpu(t, sub, r)
            _same(got, _orc(orc, sub, r), f"{name} nq = {nq} r = {r!r}")
            _model(pts, sub, r, cfg, got)
    for r in (rs[1], rs[2]):                           # 5000 queries: below P/2 (ghost pairs for one wrap)
        _same(_gpu(t, qs, r), _orc(orc, qs, r), f"{name} nq = 5000 r = {r!r}")
    # seam placements again, minus exact copies of tree points (an exact distance tie makes the nearest NODE the
    # documented tie, where device and reference may differ)
    existing = {tuple(p) for p in pts}
    extra = np.array([p for p in M.points(4, 150, cfg) if tuple(p) not in existing])
    for p in extra:
        orc.insert(p)
        t.insert(p)
    allpts = np.vstack([pts, extra])
    sub = np.ascontiguousarray(qs[:2049])
    for r in (rs[1], rs[4], rs[6]):
        got = _gpu(t, sub, r)
        _same(got, _orc(orc, sub, r), f"{name} tail r = {r!r}")
        _model(allpts, sub, r, cfg, got)
    gi, gd = t.nearest(qs)
    oi, od = orc.nearest_batch(qs, nthreads=8)
    assert np.array_equal(gd.view(np.uint64), od.view(np.uint64)) and np.array_equal(gi, oi)


@pytest.mark.parametrize("name", CONFIG_NAMES)
def test_wrapped_range_per_query_radii(ctx, name):
    """Per-query radii (always the two-pass kernel on a wrapped tree): every test radius and the degenerate
    0, -1, NaN, inf and 1e-300, mixed in one batch; a batch of equal radii gives the uniform-radius result."""
    cfg = M.CONFIGS[name]
    d, wraps, wps, _ = cfg
    pts, orc, t = _trees(ctx, cfg)
    qs = M.queries(5, 2049, cfg, pts)
    menu = np.array(M.radii(wps) + [0.0, -1.0, np.nan, np.inf, 1e-300])
    radii = np.ascontiguousarray(menu[np.arange(len(qs)) % len(menu)])
    got = _gpu(t, qs, None, ranges=radii)
    _same(got, _orc(orc, qs, ranges=radii), f"{name} per-query radii")
    _model(pts, qs, None, cfg, got, ranges=radii)
    r = M.radii(wps)[2]                                # exactly P/2: ghost pairs for the uniform call
    _same(_gpu(t, qs, None, ranges=np.full(len(qs), r)), _gpu(t, qs, r), f"{name} equal per-query radii")


@pytest.mark.parametrize("name", CONFIG_NAMES)
def test_wrapped_nearest(ctx, name):
    """Nearest at 1, 3 and 5000 queries (above the thread-per-query threshold, which wrapped trees do not take)."""
    cfg = M.CONFIGS[name]
    d, wraps, wps, _ = cfg
    pts, orc, t = _trees(ctx, cfg)
    qs = M.queries(6, 5000, cfg, pts)
    for nq in (1, 3, 5000):
        sub = np.ascontiguousarray(qs[:nq])
        gi, gd = t.nearest(sub)
        oi, od = orc.nearest_batch(sub, nthreads=8)
        assert np.array_equal(gd.view(np.uint64), od.view(np.uint64)), f"{name} nq = {nq}: distances differ"
        assert np.array_equal(gi, oi), f"{name} nq = {nq}: nodes differ"
        for qi in _sample(nq):
            mi, md = M.nearest(pts, sub[qi], wraps, wps)
            assert gi[qi] == mi and gd[qi].view(np.uint64) == np.float64(md).view(np.uint64), (name, nq, qi)


@pytest.mark.parametrize("name", CONFIG_NAMES)
def test_wrapped_nearest_tie_across_identities(ctx, name):
    """The real identity reaches A, a ghost reaches B (inserted first) at the same distance: A, as on the oracle."""
    cfg = M.CONFIGS[name]
    d, wraps, wps, _ = cfg
    pts, q, a = M.tie_tree(cfg)
    orc = oracle.KDTree(d, wraps, wps)
    orc.insert_batch(pts)
    t = DeviceTree(ctx, d, wraps=wraps, wrap_points=wps)
    t.insert_batch(pts)
    gi, gd = t.nearest(q[None, :])
    oi, od = orc.find_nearest(q)
    assert gi[0] == oi == a
    assert gd[0].view(np.uint64) == np.float64(od).view(np.uint64)


@pytest.mark.parametrize("d", [2, 3, 4])
def test_two_pass_kernel_on_unwrapped_trees(ctx, d):
    """The count / scan / fill kernel (the fall-back for trees of >= 2^27 indexed nodes), forced on plain trees:
    uniform radius and per-query radii incl. the degenerate ones, against the oracle and the single-pass kernel."""
    lo = [-20.0, -20.0, -20.0, 0.0][:d]
    hi = [20.0, 20.0, 20.0, 2 * np.pi][:d]
    pts = W.uniform_points(41, 30000, lo, hi)
    qs = W.uniform_points(42, 2500, lo, hi)
    qs[0] = pts[0]
    qs[1] = np.nan
    orc = oracle.KDTree(d)
    orc.insert_batch(pts)
    t = DeviceTree(ctx, d)
    t.insert_batch(pts)
    r = 2.2 if d == 4 else 1.1
    radii = np.ascontiguousarray(np.array([r, 0.5 * r, 3.0 * r, 0.0, -1.0, np.nan, 1e-300])[np.arange(len(qs)) % 7])
    radii[7] = np.inf                                   # one list of every node
    single = _gpu(t, qs, r)
    single_pq = _gpu(t, qs, None, ranges=radii)
    with _TwoPass(ctx):
        two = _gpu(t, qs, r)
        two_pq = _gpu(t, qs, None, ranges=radii)
    _same(two, _orc(orc, qs, r), f"d = {d} two-pass")
    _same(two, single, f"d = {d} two-pass vs single pass")
    _same(two_pq, _orc(orc, qs, ranges=radii), f"d = {d} two-pass per-query radii")
    _same(two_pq, single_pq, f"d = {d} two-pass vs single pass, per-query radii")


# ------------------------------------------------------------------------------------ consumers of wrapped trees
def test_extend_query_refuses_wrapped_trees(ctx, building2):
    pts = M.points(1, 500, M.CONFIGS["testGhost_z"])
    t = DeviceTree(ctx, 3, wraps=[2], wrap_points=[2 * np.pi])
    t.insert_batch(pts)
    centers, radii, _ = building2
    S = SphereSet(ctx, centers, radii)
    with pytest.raises(A.RRTQXError) as e:
        extend_query(t, S, pts[3] + 0.01, 1.0, 0.5, 0)
    assert e.value.status == A.ERR_UNSUPPORTED


def test_sweep_2d_refuses_two_wrap_dimensions(ctx):
    pts = M.points(1, 300, M.CONFIGS["three_wraps"])
    t = DeviceTree(ctx, 4, wraps=[0, 3], wrap_points=[3.0, 2 * np.pi])
    t.insert_batch(pts)
    E = EdgeSet(t)
    src = np.arange(1, 300, dtype=np.int32)
    E.upload(src, src - 1, np.r_[-1, src - 1].astype(np.int32))
    E.solve_trajectories(1.0)
    P = PolygonSet(ctx)
    P.upload([("ball", (1.0, 1.0), 0.5)])
    with pytest.raises(A.RRTQXError) as e:
        E.add_sweep_2d(P, [0], 0.5, 5.0, 1.0)
    assert e.value.status == A.ERR_INVALID


def test_reparenting_invalidates_dubins_trajectories(ctx):
    """Parent edges re-pointed after the trajectories were solved make the sweeps refuse (their resident
    trajectories are the old edges'); clearing parents does not.  Both states are checked against the oracle."""
    from test_gpu_sweep2d import (DELTA, R_TURN, RHO, _csr, _dubins_graph, _oracle_add, _orc_obstacles,
                                  _reference_polygons)
    n = 4000
    pts, t, src, dst, parent = _dubins_graph(ctx, n, 4.0, seed=17)
    P = PolygonSet(ctx)
    obstacles = _reference_polygons("ref_rand_Static.txt")
    P.upload(obstacles)
    orc_obs = _orc_obstacles(P)
    orc = oracle.KDTree(4, (3,), (2 * math.pi,))
    orc.insert_batch(pts)
    row_ptr = _csr(src, n)
    picks = list(range(0, len(obstacles), 4))

    def check(par):
        tptr, txy = E.trajectories()
        hits = 0
        for o in picks:
            ge, gn = E.add_sweep_2d(P, [o], RHO, DELTA, R_TURN).fetch()
            wb, wo, _ = _oracle_add(orc, orc_obs[o], pts, row_ptr, dst, par, tptr, txy)
            assert set(ge.tolist()) == wb and len(ge) == len(wb), o
            assert set(gn.tolist()) == wo and len(gn) == len(wo), o
            hits += len(wo)
        return hits

    E = EdgeSet(t)
    E.upload(src, dst)                                  # no parents yet
    E.solve_trajectories(R_TURN)
    E.set_parents(np.arange(n, dtype=np.int32), parent)  # the first parents are new parent edges
    with pytest.raises(A.RRTQXError) as e:
        E.add_sweep_2d(P, [0], RHO, DELTA, R_TURN)
    assert e.value.status == A.ERR_STATE
    E.solve_trajectories(R_TURN)
    assert check(parent) > 0

    cleared = np.nonzero(parent >= 0)[0][::9].astype(np.int32)
    par1 = parent.copy()
    par1[cleared] = -1
    E.set_parents(cleared, np.full(len(cleared), -1, dtype=np.int32))
    check(par1)                                         # still valid: items without a parent edge are never read

    # re-point 50 nodes to another of their neighbours
    movable = [v for v in range(1, n) if par1[v] >= 0 and np.count_nonzero(src == v) >= 2][:50]
    assert len(movable) == 50
    par2 = par1.copy()
    for v in movable:
        nb = dst[src == v]
        par2[v] = int(nb[nb != par1[v]][0])
    E.set_parents(np.array(movable, dtype=np.int32), par2[movable])
    with pytest.raises(A.RRTQXError) as e:
        E.add_sweep_2d(P, [0], RHO, DELTA, R_TURN)
    assert e.value.status == A.ERR_STATE
    E.solve_trajectories(R_TURN)
    tptr, _ = E.trajectories()
    assert len(tptr) == len(src) + n + 1
    check(par2)
