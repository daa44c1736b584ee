"""rrtqx_extend_query_dubins_multi: one iteration of many independent Dubins planners (config C4's [x y t theta]
tree with the heading wrapped at 2 pi, among 2-D polygons) in one call.  Every instance must see exactly what
rrtqx_extend_query_dubins gives it, trajectory rows included, and the lock-step replay must match the oracle."""
import ctypes as C
import math

import numpy as np
import pytest

import oracle
from rrtqx_3d_b200 import _abi as A
from rrtqx_3d_b200 import workloads as W
from rrtqx_3d_b200.device import (Context, DeviceTree, DubinsResult, PolygonSet, extend_query_dubins,
                                  extend_query_dubins_multi, insert_multi)
from test_gpu_collision import _orc_obstacles_2d
from test_gpu_extend_dubins import (R_TURN, RHO, ROOT, ROOT_REF, TWO_PI, _bits, _check_ball, _check_edges,
                                    _check_nearest, _samples, _tree, _world)

pytestmark = pytest.mark.gpu


class _Slice:
    """One instance's part of the shared trajectory result, in the shape _check_edges reads."""

    def __init__(self, fetched, first, n_edges):
        dist, typ, ptr, xy = fetched
        self.parts = (dist[first:first + n_edges], typ[first:first + n_edges],
                      ptr[first:first + n_edges + 1] - ptr[first], xy[ptr[first]:ptr[first + n_edges]])

    def fetch(self):
        return self.parts


def _sliced(res, fetched):
    """res with .trajectories replaced by its slice of the packed result (a shallow copy)."""
    out = type(res)()
    for k in type(res).__slots__:
        setattr(out, k, getattr(res, k))
    out.trajectories = _Slice(fetched, res.first_edge, len(res.edge_dist))
    return out


def _per_node(res, fetched):
    """node -> (key bits, (dist bits, type, collide, row bits) of edge new -> node, the same of node -> new)."""
    _, _, ptr, xy = fetched
    f = res.first_edge
    out = {}
    for k, node in enumerate(res.idx.tolist()):
        edges = []
        for e in (2 * k, 2 * k + 1):
            rows = xy[ptr[f + e]:ptr[f + e + 1]]
            edges.append((int(_bits([res.edge_dist[e]])[0]), int(res.edge_type[e]), int(res.edge_collide[e]),
                          _bits(rows.reshape(-1)).tobytes()))
        out[node] = (int(_bits([res.dist[k]])[0]), edges[0], edges[1])
    return out


def _same(multi, mf, single, sf, capacity):
    """Multi result equals the single call's bit for bit; with a capacity below the count, its neighbours are any
    `capacity` of the single call's complete ball, each with the same key, edges and rows."""
    assert (multi.nearest_idx, _bits([multi.nearest_dist])[0], multi.count) == \
        (single.nearest_idx, _bits([single.nearest_dist])[0], single.count)
    assert np.array_equal(_bits(multi.point), _bits(single.point))
    a, b = _per_node(multi, mf), _per_node(single, sf)
    if capacity < single.count:
        assert len(a) == capacity and all(a[k] == b[k] for k in a)
    else:
        assert a == b


# ------------------------------------------------------------------------ 1. lock-step replay against the oracle
def test_lockstep_replay_matches_oracle(ctx):
    """8 instances (seeds 1..8), 1500 lock-step rounds: 4 city-block instances (r 1.06, delta 1: two share the set,
    one has every other block inactive, one an empty set) and 4 paper-regime instances (delta 10, gamma 100, r = 10 >
    pi, a reference polygon file plus balls, one set shared by all four).  delta is one value per call, so each
    regime is one multi call per round; the accepted samples of both go to one insert_multi."""
    n_iter = 1500
    P_city, orc_city = _world(ctx, "city")
    P_ref, orc_ref = _world(ctx, "ref")
    blocks = W.c4_city_blocks()
    half = (np.arange(len(blocks)) % 2).astype(np.uint8)
    P_half = PolygonSet(ctx)
    P_half.upload(blocks, active=half)
    P_empty = PolygonSet(ctx)
    P_empty.upload([])
    city_sets = [P_city, P_city, P_half, P_empty]
    city_orc = [(orc_city, None), (orc_city, None), (orc_city, half), ([], None)]
    samples = [_samples(1 + i, n_iter) for i in range(8)]
    roots = [ROOT] * 4 + [ROOT_REF] * 4
    trees, orcs = zip(*[_tree(ctx) for _ in range(8)])
    trees, orcs = list(trees), list(orcs)
    assert insert_multi(trees, np.stack(roots)).tolist() == [0] * 8
    for o, r in zip(orcs, roots):
        o.insert(r)
    pts = np.zeros((8, n_iter + 1, 4))
    pts[:, 0] = roots
    sizes = [1] * 8
    traj = DubinsResult(ctx)
    n_edges = [0, 0]
    n_ties = [0]
    for it in range(n_iter):
        q = np.stack([s[it] for s in samples])
        n_paper = sizes[4:]
        r_paper = [min(100.0 * (math.log(n) / n) ** 0.25, 10.0) if n > 1 else 10.0 for n in n_paper]
        groups = ((range(4), city_sets, [1.06] * 4, 1.0), (range(4, 8), [P_ref] * 4, r_paper, 10.0))
        accepted, acc_pts = [], []
        for g, (ids, sets, ranges, delta) in enumerate(groups):
            res = extend_query_dubins_multi([trees[i] for i in ids], sets, q[list(ids)], ranges, RHO, R_TURN,
                                            delta=delta, flags=A.EXTEND_SATURATE, capacity=1024, trajectories=traj)
            fetched = traj.fetch()
            for k, i in enumerate(ids):
                rk, P = res[k], pts[i, :sizes[i]]
                _check_nearest(orcs[i], P, q[i], rk)
                want_p = oracle.saturate_dubins(q[i], P[rk.nearest_idx], delta)
                assert np.array_equal(_bits(rk.point), _bits(want_p)), (it, i)
                _check_ball(orcs[i], rk, ranges[k])
                if g == 0 or it < 50 or it % 25 == 0:
                    obs, active = city_orc[k] if g == 0 else (orc_ref, None)
                    _check_edges(_sliced(rk, fetched), P, obs, active=active, n_ties=n_ties)
                    n_edges[g] += 2 * rk.count
                fwd_ok = (rk.edge_collide[0::2] == 0) & np.isfinite(rk.edge_dist[0::2])
                if fwd_ok.any():
                    accepted.append(i)
                    acc_pts.append(rk.point)
        if accepted:
            got = insert_multi([trees[i] for i in accepted], np.stack(acc_pts))
            assert got.tolist() == [orcs[i].insert(p) for i, p in zip(accepted, acc_pts)]
            for i, p in zip(accepted, acc_pts):
                pts[i, sizes[i]] = p
                sizes[i] += 1
    for t, o in zip(trees, orcs):
        assert len(t) == len(o) > 1
        for a, b in zip(t.kd_fields(), o.fields()):
            assert np.array_equal(a, b)
    # the paper-regime trees crossed the re-index threshold (64 unsorted nodes): their queries ran on the grid index
    assert min(sizes[4:]) > 65, sizes
    assert n_edges[0] > 500 and n_edges[1] > 3000, n_edges
    assert n_ties[0] <= max(1, sum(n_edges) // 200)


# ------------------------------------------------------------------------ 2. multi equals single, bit for bit
def _mixed_trees(ctx):
    """A root-only tree, a 40-pose tree in the unsorted tail, 3000 poses, and a 2e5-pose C4 tree."""
    t0, _ = _tree(ctx, ROOT[None, :])
    t1, _ = _tree(ctx)
    tail = _samples(61, 40)
    for p in tail:
        t1.insert(p)
    p2 = _samples(62, 3000)
    p2[1, 3], p2[2, 3], p2[3, 3] = 0.0, math.pi, np.nextafter(TWO_PI, 0.0)
    t2, _ = _tree(ctx, p2)
    p3 = _samples(63, 200_000)
    t3, _ = _tree(ctx, p3)
    return [t0, t1, t2, t3], [ROOT[None, :], tail, p2, p3]


def test_multi_equals_single(ctx):
    trees, pts = _mixed_trees(ctx)
    blocks = W.c4_city_blocks()
    P = PolygonSet(ctx)
    P.upload(blocks, active=(np.arange(len(blocks)) % 3 != 0).astype(np.uint8))
    base = np.array([[0.3, -0.2, 0.0, 0.0], [3.0, -4.0, 0.0, 0.0], [0.5, 0.5, 0.0, 0.0], [1.5, 2.5, 0.0, 0.0]])
    rounds = []
    for th in (0.0, math.pi, np.nextafter(math.pi, 4.0), np.nextafter(TWO_PI, 0.0), TWO_PI):
        for r in (0.0, -1.0, float("nan"), math.pi, np.nextafter(math.pi, 4.0), float("inf")):
            q = base.copy()
            q[:, 3] = th
            rounds.append((q, [r, r, r if r != float("inf") else 6.0, r if r != float("inf") else 1.06]))
    on_node = np.stack([pts[0][0], pts[1][7], pts[2][17], pts[3][1234]])
    far = np.array([[1e4, -3e4, 0.0, 2.0]] * 4)
    rounds += [(on_node, [1.06, 2.5, 1.06, 1.06]), (far, [1.06, 4.0, 2.5, 1.06]), (base, [2.0, 6.0, 4.0, 2.5])]
    seen = {"edges": 0, "collide": 0, "partial": 0}
    mtraj, straj = DubinsResult(ctx), DubinsResult(ctx)
    for flags in (A.EXTEND_SATURATE, 0, A.CHECK_IGNORE_ACTIVE, A.EXTEND_SATURATE | A.CHECK_IGNORE_ACTIVE):
        for q, ranges in rounds:
            single, sfetch = [], []
            for i in range(4):
                s = extend_query_dubins(trees[i], P, q[i], ranges[i], RHO, R_TURN, delta=1.5, flags=flags,
                                        capacity=8192, trajectories=straj)
                single.append(s)
                sfetch.append(straj.fetch())
            for cap in (8192, 0, 5):
                got = extend_query_dubins_multi(trees, [P] * 4, q, ranges, RHO, R_TURN, delta=1.5, flags=flags,
                                                capacity=cap, trajectories=mtraj)
                mf = mtraj.fetch()
                assert mtraj.sizes()[0] == sum(2 * min(s.count, cap) for s in single)
                for i in range(4):
                    _same(got[i], mf, single[i], sfetch[i], cap)
                    seen["partial"] += cap < single[i].count
            seen["edges"] += sum(2 * s.count for s in single)
            seen["collide"] += sum(int(s.edge_collide.sum()) for s in single)
    assert seen["edges"] > 10000 and seen["collide"] > 0 and seen["partial"] > 0, seen
    # without a trajectory handle the results are the same
    got = extend_query_dubins_multi(trees, [P] * 4, base, [2.0, 6.0, 4.0, 2.5], RHO, R_TURN, delta=1.5)
    for i in range(4):
        s = extend_query_dubins(trees[i], P, base[i], [2.0, 6.0, 4.0, 2.5][i], RHO, R_TURN, delta=1.5)
        assert (got[i].count, got[i].nearest_idx) == (s.count, s.nearest_idx)
        assert np.array_equal(np.sort(got[i].idx), np.sort(s.idx))


# ------------------------------------------------------------------------ 3. row-scratch regrowth
def test_row_scratch_regrowth():
    """A fresh context: the first multi call's rows exceed the initial scratch (16384 rows); the call grows it and
    repeats once (6 launches), the next one fits (3 launches); results equal the single calls."""
    c = Context(0)
    P, _ = _world(c, "city")
    trees = [_tree(c, _samples(70 + i, 400))[0] for i in range(3)]
    q = np.array([[0.0, 0.0, 0.0, 1.0], [1.0, 2.0, 0.0, 4.0], [-3.0, 5.0, 0.0, 6.0]])
    ranges = [float("inf")] * 3
    single = [extend_query_dubins(t, P, q[i], ranges[i], RHO, R_TURN, trajectories=True) for i, t in enumerate(trees)]
    sf = [s.trajectories.fetch() for s in single]
    traj = DubinsResult(c)
    for attempt, launches in ((0, 6), (1, 3)):
        k0 = c.kernel_launches()
        got = extend_query_dubins_multi(trees, [P] * 3, q, ranges, RHO, R_TURN, capacity=512, trajectories=traj)
        assert c.kernel_launches() - k0 == launches, attempt
        assert traj.sizes()[1] > 16384
        mf = traj.fetch()
        for i in range(3):
            _same(got[i], mf, single[i], sf[i], 512)


# ------------------------------------------------------------------------ 4. more instances than SMs
def test_more_instances_than_sms(ctx):
    P, _ = _world(ctx, "city")
    rng = np.random.default_rng(300)
    n = 300
    trees = [_tree(ctx, _samples(1000 + i, int(rng.integers(1, 400))))[0] for i in range(n)]
    mtraj, straj = DubinsResult(ctx), DubinsResult(ctx)
    for rnd in range(2):
        q = _samples(2000 + rnd, n)
        ranges = rng.uniform(1.0, 8.0, n)
        got = extend_query_dubins_multi(trees, [P] * n, q, ranges, RHO, R_TURN, delta=1.0, flags=A.EXTEND_SATURATE,
                                        trajectories=mtraj)
        mf = mtraj.fetch()
        for i in range(n):
            s = extend_query_dubins(trees[i], P, q[i], ranges[i], RHO, R_TURN, delta=1.0, flags=A.EXTEND_SATURATE,
                                    trajectories=straj)
            _same(got[i], mf, s, straj.fetch(), 1024)
        insert_multi(trees, np.stack([g.point for g in got]))


# ------------------------------------------------------------------------ 5. launch counts
def test_steady_state_launch_counts(ctx):
    P, _ = _world(ctx, "city")
    n = 16
    trees = []
    for i in range(n):
        t, _ = _tree(ctx, _samples(80 + i, 3000))
        t.reindex()
        trees.append(t)
    traj = DubinsResult(ctx)
    extend_query_dubins_multi(trees, [P] * n, _samples(99, n), np.full(n, 2.0), RHO, R_TURN, trajectories=traj)
    for k in range(5):
        q = _samples(100 + k, n)
        k0 = ctx.kernel_launches()
        got = extend_query_dubins_multi(trees, [P] * n, q, np.full(n, 2.0), RHO, R_TURN, delta=1.0,
                                        flags=A.EXTEND_SATURATE, trajectories=traj)
        k1 = ctx.kernel_launches()
        insert_multi(trees, np.stack([g.point for g in got]))
        k2 = ctx.kernel_launches()
        assert (k1 - k0, k2 - k1) == (3, 1)
    k0 = ctx.kernel_launches()
    assert ctx.L.rrtqx_extend_query_dubins_multi(None, None, 0, None, None, 1.0, RHO, R_TURN, 0, 0,
                                                 *([None] * 9)) == A.OK
    assert extend_query_dubins_multi([], [], np.zeros((0, 4)), [], RHO, R_TURN) == []
    assert ctx.kernel_launches() == k0


# ------------------------------------------------------------------------ 6. interleaving and state
def test_interleaved_single_and_multi_and_polygon_updates(ctx):
    rng = np.random.default_rng(9)
    n = 6
    trees = [_tree(ctx, _samples(120 + i, 2000))[0] for i in range(n)]
    blocks = W.c4_city_blocks()
    active = np.ones(len(blocks), np.uint8)
    P_toggle, P_fixed = PolygonSet(ctx), PolygonSet(ctx)
    P_toggle.upload(blocks, active=active)
    P_fixed.upload(blocks)
    sets = [P_toggle, P_fixed] * (n // 2)
    kept, mtraj = DubinsResult(ctx), DubinsResult(ctx)
    for rnd in range(12):
        q = _samples(140 + rnd, n)
        ranges = rng.uniform(1.5, 4.0, n)
        # a single call's result, then a multi call on the same trees: the single result must stay as it was
        s0 = extend_query_dubins(trees[0], sets[0], q[0], ranges[0], RHO, R_TURN, trajectories=kept)
        before = kept.fetch()
        multi = extend_query_dubins_multi(trees, sets, q, ranges, RHO, R_TURN, trajectories=mtraj)
        after = kept.fetch()
        assert all(np.array_equal(_bits(a) if a.dtype == np.float64 else a, _bits(b) if b.dtype == np.float64 else b)
                   for a, b in zip(before, after))
        mf = mtraj.fetch()
        _same(multi[0], mf, s0, before, 1024)
        for i in range(n):
            s = extend_query_dubins(trees[i], sets[i], q[i], ranges[i], RHO, R_TURN, trajectories=True)
            _same(multi[i], mf, s, s.trajectories.fetch(), 1024)
        again = extend_query_dubins_multi(trees, sets, q, ranges, RHO, R_TURN, trajectories=mtraj)
        af = mtraj.fetch()
        for a, b in zip(again, multi):
            _same(a, af, b, mf, 1024)
        # toggle blocks of the shared set between rounds: the instances that use it see the change
        active[rng.integers(len(blocks), size=10)] ^= 1
        P_toggle.upload(blocks, active=active)
        probe = extend_query_dubins_multi(trees, sets, q, np.full(n, 6.0), RHO, R_TURN, trajectories=mtraj)
        pf = mtraj.fetch()
        orc_obs = _orc_obstacles_2d(P_fixed)
        for i in range(n):
            P_i = np.asarray(trees[i].positions())
            _check_edges(_sliced(probe[i], pf), P_i, orc_obs, active=active if sets[i] is P_toggle else None)
        if rnd % 3 == 2:
            insert_multi(trees, _samples(160 + rnd, n))
    assert not active.all()


# ------------------------------------------------------------------------ 7. refusals
def _raw_multi(ctx, trees, sets, pts, ranges, capacity=64):
    """The C call with sentinel-filled outputs and a copy of the points; returns (status, message, outputs, whether
    the points changed, the trajectory handle)."""
    n = len(trees)
    th = (A.vp * n)(*[None if t is None else t.h for t in trees])
    ph = (A.vp * n)(*[None if s is None else s.h for s in sets])
    w = n * 64
    outs = [np.full(n, -7, np.int32), np.full(n, -7.0), np.full(n, -7, np.int32), np.full(w, -7, np.int32),
            np.full(w, -7.0), np.full(2 * w, -7.0), np.full(2 * w, -7, np.int32), np.full(2 * w, 7, np.uint8)]
    p = np.array(pts, copy=True) if isinstance(pts, np.ndarray) else pts
    res = A.vp()
    st = ctx.L.rrtqx_extend_query_dubins_multi(th, ph, n, A.ptr(p) if isinstance(p, np.ndarray) else p,
                                               A.ptr(ranges), 1.0, RHO, R_TURN, A.EXTEND_SATURATE, capacity,
                                               *[A.ptr(o) for o in outs], C.byref(res))
    msg = (ctx.L.rrtqx_last_error(ctx.h) or b"").decode()
    moved = isinstance(p, np.ndarray) and not np.array_equal(p, pts)
    made = bool(res.value)
    if made:
        ctx.L.rrtqx_dubins_result_destroy(res)
    return st, msg, outs, moved, made


def _untouched(outs):
    return all(np.all(o == (7 if o.dtype == np.uint8 else -7)) for o in outs)


def test_refusals(ctx):
    P, _ = _world(ctx, "city")
    good = [_tree(ctx, _samples(170, 500))[0], _tree(ctx, _samples(171, 500))[0]]
    pts, ranges = _samples(172, 2), np.array([2.0, 2.0])

    def ok_after():
        st, msg, outs, moved, made = _raw_multi(ctx, good, [P, P], pts, ranges)
        assert st == A.OK, msg
        assert not _untouched(outs) and made

    ctx2 = Context(0)
    other, _ = _tree(ctx2, _samples(173, 100))
    P_other, _ = _world(ctx2, "city")

    def bad_tree(d, **kw):
        t = DeviceTree(ctx, d, **kw)
        t.insert_batch(_samples(174, 100)[:, :d])
        return t

    empty, _ = _tree(ctx)
    cases = [
        ([good[0], None], [P, P], A.ERR_INVALID, "instance 1"),
        ([good[0], good[1]], [P, None], A.ERR_INVALID, "instance 1"),
        ([good[0], other], [P, P], A.ERR_INVALID, "another context"),
        ([good[0], good[1]], [P, P_other], A.ERR_INVALID, "another context"),
        ([good[0], good[0]], [P, P], A.ERR_INVALID, "twice"),
        ([good[0], bad_tree(3, wraps=(2,), wrap_points=(TWO_PI,))], [P, P], A.ERR_UNSUPPORTED, "instance 1"),
        ([bad_tree(4, wraps=(0,), wrap_points=(TWO_PI,)), good[1]], [P, P], A.ERR_UNSUPPORTED, "instance 0"),
        ([good[0], bad_tree(4, wraps=(3,), wrap_points=(2 * 3.14159,))], [P, P], A.ERR_UNSUPPORTED, "instance 1"),
        ([good[0], bad_tree(4)], [P, P], A.ERR_UNSUPPORTED, "instance 1"),
        ([empty, good[1]], [P, P], A.ERR_EMPTY_TREE, "instance 0"),
    ]
    for trees, sets, status, words in cases:
        k0 = ctx.kernel_launches()
        st, msg, outs, moved, made = _raw_multi(ctx, trees, sets, pts, ranges)
        assert st == status and words in msg, (st, msg, words)
        assert _untouched(outs) and not moved and not made, words
        assert ctx.kernel_launches() == k0
        ok_after()
    st, msg, outs, moved, made = _raw_multi(ctx, good, [P, P], pts, ranges, capacity=-1)
    assert st == A.ERR_INVALID and "capacity" in msg and _untouched(outs) and not moved and not made
    ok_after()
    import torch
    dpts = torch.tensor(pts, device="cuda")
    st, msg, outs, moved, made = _raw_multi(ctx, good, [P, P], int(dpts.data_ptr()), ranges)
    assert st == A.ERR_INVALID and "host array" in msg and _untouched(outs) and not made
    ok_after()
    dr = torch.tensor(ranges, device="cuda")
    th = (A.vp * 2)(good[0].h, good[1].h)
    ph = (A.vp * 2)(P.h, P.h)
    p = np.array(pts, copy=True)
    st = ctx.L.rrtqx_extend_query_dubins_multi(th, ph, 2, A.ptr(p), int(dr.data_ptr()), 1.0, RHO, R_TURN,
                                               A.EXTEND_SATURATE, 64, *([None] * 9))
    assert st == A.ERR_INVALID and np.array_equal(p, pts)
    ok_after()
