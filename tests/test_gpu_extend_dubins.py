"""Config C4 (DubinsEdge, [x y t theta] with the heading wrapped at 2 pi): the fused per-iteration call
rrtqx_extend_query_dubins (nearest -> saturate -> ball -> calculateTrajectory + explicitEdgeCheck of both edges per
neighbour) against the oracle on grown trees, bit for bit against the same work composed from the batch entry
points, at the input edges, and its refusals."""
import ctypes as C
import math
import os

import numpy as np
import pytest

import oracle
import wrap_model as WM
from rrtqx_3d_b200 import _abi as A
from rrtqx_3d_b200 import workloads as W
from rrtqx_3d_b200.device import (DeviceTree, DubinsResult, PolygonSet, SphereSet, extend_query,
                                  extend_query_dubins, extend_query_dubins_composed)
from rrtqx_3d_b200.formats import read_polygon_obstacles

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TWO_PI = 2.0 * math.pi
RHO, R_TURN = 0.5, 1.0
TOL = 1e-9
ROOT = np.array([0.0, 0.0, 0.0, 1.0])
ROOT_REF = np.array([10.0, 0.0, 0.0, 1.0])   # a pose in free space of ref_rand_Static (the origin is inside a polygon)


def _tree(ctx, pts=None):
    t = DeviceTree(ctx, 4, wraps=(3,), wrap_points=(TWO_PI,))
    orc = oracle.KDTree(4, wraps=[3], wrap_points=[TWO_PI])
    if pts is not None:
        t.insert_batch(pts)
        orc.insert_batch(pts)
    return t, orc


def _samples(seed, n):
    return W.uniform_points(seed, n, [-50.0, -50.0, 0.0, 0.0], [50.0, 50.0, 0.0, TWO_PI])


def _world(ctx, which):
    if which == "city":
        obstacles = W.c4_city_blocks()
    else:
        obs = read_polygon_obstacles(os.path.join(GOLDEN, "ref_rand_Static.txt"))
        obstacles = [("polygon", o["polygon"]) for o in obs]
        obstacles += [("ball", (5.0, 5.0), 3.0), ("ball", (-20.0, 31.0), 4.0), ("ball", (30.0, -12.0), 2.5)]
    P = PolygonSet(ctx)
    P.upload(obstacles)
    from test_gpu_collision import _orc_obstacles_2d
    return P, _orc_obstacles_2d(P)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _check_ball(orc, res, r):
    oi, ok = orc.find_within_range(r, res.point)
    orc.empty(oi)
    o, g = np.argsort(oi), np.argsort(res.idx)
    assert res.count == len(oi)
    assert np.array_equal(res.idx[g], oi[o])
    assert np.array_equal(_bits(res.dist[g]), _bits(ok[o]))


def _check_edges(res, pts, orc_obs, active=None, n_ties=None):
    """Per-edge Dubins length / word / rows against the oracle, collision against orc_edge_check_dubins run on the
    device rows, OR-ed over the (active) obstacles."""
    L = oracle.lib()
    f = lambda a: oracle._p(np.ascontiguousarray(a, dtype=np.float64), oracle.c_f64p)
    dist, typ, ptr, xy = res.trajectories.fetch()
    m = len(res.idx)
    assert len(dist) == 2 * m and ptr[-1] == len(xy)
    assert np.array_equal(_bits(dist), _bits(res.edge_dist)) and np.array_equal(typ, res.edge_type)
    ties = 0
    for e in range(2 * m):
        nb = pts[res.idx[e >> 1]]
        s, g = (res.point, nb) if e % 2 == 0 else (nb, res.point)
        od, ot, otr = oracle.dubins_trajectory(s, g, R_TURN)
        rows = xy[ptr[e]:ptr[e + 1]]
        if ot != typ[e]:   # admissible only under a length tie between two words (different libm, last ulp)
            assert od == dist[e] or abs(od - dist[e]) <= TOL * max(1.0, abs(od)), (e, ot, typ[e], od, dist[e])
            ties += 1
        else:
            if math.isnan(od) or math.isinf(od):
                assert (math.isnan(od) and math.isnan(dist[e])) or od == dist[e], (e, od, dist[e])
            else:
                assert abs(od - dist[e]) <= TOL * max(1.0, abs(od)), (e, od, dist[e])
            assert len(rows) == len(otr), (e, len(rows), len(otr))
            fin = np.isfinite(otr)
            assert np.array_equal(np.isfinite(rows), fin)
            assert np.all(np.abs(rows[fin] - otr[fin]) <= TOL * np.maximum(1.0, np.abs(otr[fin]))), e
        want = 0
        for k, ob in enumerate(orc_obs):
            if active is not None and not active[k]:
                continue
            if L.orc_edge_check_dubins(C.byref(ob), f(s[:2]), f(g[:2]), f(rows), len(rows), RHO, R_TURN):
                want = 1
                break
        assert res.edge_collide[e] == want, (e, res.edge_collide[e], want)
    if n_ties is not None:
        n_ties[0] += ties
    return ties


def _order(res):
    """Neighbours in ascending node order, and their edges (2i, 2i+1) in that order: lists are sets."""
    g = np.argsort(res.idx, kind="stable")
    return g, np.stack([2 * g, 2 * g + 1], axis=1).reshape(-1)


def _check_nearest(orc, pts, q, res):
    wi, wd = WM.nearest(pts, q, [3], [TWO_PI])
    _, od = orc.find_nearest(q)
    assert res.nearest_idx == wi and _bits([res.nearest_dist])[0] == _bits([wd])[0]
    assert _bits([res.nearest_dist])[0] == _bits([od])[0]


@pytest.mark.parametrize("regime", ["c4", "paper"])
def test_c4_replay_matches_oracle(ctx, regime):
    """Grow a tree from one pose for 3000 iterations with RRTQX_EXTEND_SATURATE: c4 = r 1.06 (delta 1.0) among the
    city blocks, paper = delta 10, gamma 100 (r = 10 > pi) among a reference polygon file plus balls."""
    P, orc_obs = _world(ctx, "city" if regime == "c4" else "ref")
    n_iter = 3000
    samples = _samples(11 if regime == "c4" else 12, n_iter)
    root = ROOT if regime == "c4" else ROOT_REF
    t, orc = _tree(ctx, root[None, :])
    pts = np.zeros((n_iter + 1, 4))
    pts[0] = root
    n = 1
    traj = DubinsResult(ctx)
    n_ties, n_edges, n_inserted = [0], 0, 0
    for it in range(n_iter):
        if regime == "c4":
            delta, r = 1.0, 1.06
        else:
            delta = 10.0
            r = min(100.0 * (math.log(n) / n) ** 0.25, delta) if n > 1 else delta
        q = samples[it]
        res = extend_query_dubins(t, P, q, r, RHO, R_TURN, delta=delta, flags=A.EXTEND_SATURATE, capacity=8192,
                                  trajectories=traj)
        _check_nearest(orc, pts[:n], q, res)
        want_p = oracle.saturate_dubins(q, pts[res.nearest_idx], delta)   # driven by the node the device chose
        assert np.array_equal(_bits(res.point), _bits(want_p)), (it, res.point, want_p)
        _check_ball(orc, res, r)
        if regime == "c4" or it < 50 or it % 25 == 0:   # c4 balls hold one or two nodes: check every iteration
            _check_edges(res, pts, orc_obs, n_ties=n_ties)
            n_edges += 2 * res.count
        fwd_ok = (res.edge_collide[0::2] == 0) & np.isfinite(res.edge_dist[0::2])
        if fwd_ok.any():   # findBestParent stand-in: some forward edge is free and has a finite length
            t.insert(res.point)
            orc.insert(res.point)
            pts[n] = res.point
            n += 1
            n_inserted += 1
    # the replay must grow a tree and check many edges (seeded: 289 inserts / 6032 edges among the city blocks,
    # 1794 inserts in the reference world)
    assert n_inserted > (200 if regime == "c4" else 1000), n_inserted
    assert n_edges > 3000, n_edges
    assert n_ties[0] <= max(1, n_edges // 200)


def test_fused_equals_composed(ctx):
    """600 samples on a 20k-pose tree with an unsorted tail: the fused call and the five batch calls agree bit for
    bit (nearest, saturated point, neighbour keys, per-edge length / word / collision and every trajectory row)."""
    P, _ = _world(ctx, "city")
    pts = _samples(21, 20000)
    t, _ = _tree(ctx, pts)
    extra = _samples(22, 300)
    for p in extra:
        t.insert(p)
    allpts = np.concatenate([pts, extra])
    q = _samples(23, 600)
    fr, cr = DubinsResult(ctx), DubinsResult(ctx)
    total = 0
    for i in range(len(q)):
        r = (1.06, 2.5, 4.0)[i % 3]
        fl = A.EXTEND_SATURATE if i % 2 == 0 else 0
        a = extend_query_dubins(t, P, q[i], r, RHO, R_TURN, delta=2.0, flags=fl, trajectories=fr)
        b = extend_query_dubins_composed(t, P, q[i], r, RHO, R_TURN, allpts, delta=2.0, flags=fl, trajectories=cr)
        assert (a.nearest_idx, _bits([a.nearest_dist])[0]) == (b.nearest_idx, _bits([b.nearest_dist])[0])
        assert np.array_equal(_bits(a.point), _bits(b.point)) and a.count == b.count
        (ga, ea), (gb, eb) = _order(a), _order(b)
        assert np.array_equal(a.idx[ga], b.idx[gb]) and np.array_equal(_bits(a.dist[ga]), _bits(b.dist[gb]))
        assert np.array_equal(_bits(a.edge_dist[ea]), _bits(b.edge_dist[eb]))
        assert np.array_equal(a.edge_type[ea], b.edge_type[eb])
        assert np.array_equal(a.edge_collide[ea], b.edge_collide[eb])
        _, _, pa, xa = fr.fetch()
        _, _, pb, xb = cr.fetch()
        for e1, e2 in zip(ea, eb):
            assert np.array_equal(_bits(xa[pa[e1]:pa[e1 + 1]]), _bits(xb[pb[e2]:pb[e2 + 1]])), (i, e1)
        total += a.count
    assert total > 3000


def _full_check(t, orc, pts, P, orc_obs, q, r, delta=1.0, flags=A.EXTEND_SATURATE, capacity=8192, active=None):
    res = extend_query_dubins(t, P, q, r, RHO, R_TURN, delta=delta, flags=flags, capacity=capacity, trajectories=True)
    _check_nearest(orc, pts, q, res)
    if flags & A.EXTEND_SATURATE:
        want_p = oracle.saturate_dubins(q, pts[res.nearest_idx], delta)
    else:
        want_p = np.asarray(q, dtype=np.float64)
    assert np.array_equal(_bits(res.point), _bits(want_p))
    if capacity >= res.count:
        _check_ball(orc, res, r)
    _check_edges(res, pts, orc_obs, active=active)
    return res


def test_edge_inputs(ctx):
    P, orc_obs = _world(ctx, "city")
    pts = _samples(31, 3000)
    pts[1, 3], pts[2, 3], pts[3, 3] = 0.0, math.pi, np.nextafter(TWO_PI, 0.0)
    t, orc = _tree(ctx, pts)
    base = np.array([3.0, -4.0, 0.0, 0.0])
    # headings at the seam and at pi
    for th in (0.0, math.pi, np.nextafter(math.pi, 4.0), np.nextafter(TWO_PI, 0.0), TWO_PI):
        q = base.copy()
        q[3] = th
        for fl in (A.EXTEND_SATURATE, 0):
            _full_check(t, orc, pts, P, orc_obs, q, 2.5, delta=1.5, flags=fl)
    # radii: empty, negative, NaN, pi and the next double (the ghost's bound), +inf on a small tree
    small_pts = _samples(32, 300)
    ts, os_ = _tree(ctx, small_pts)
    for r in (0.0, -1.0, float("nan"), math.pi, np.nextafter(math.pi, 4.0), float("inf")):
        res = _full_check(ts, os_, small_pts, P, orc_obs, np.array([1.0, 2.0, 0.0, 6.0]), r, delta=3.0)
        if r == float("inf"):
            assert res.count == len(small_pts)
        if not (r > 0.0):
            assert res.count <= 1
    # a sample far outside the grid: empty ball, nearest still right
    res = _full_check(t, orc, pts, P, orc_obs, np.array([1e4, -3e4, 0.0, 2.0]), 1.06, flags=0)
    assert res.count == 0
    # a sample on an existing node: zero-length edges to it
    res = _full_check(t, orc, pts, P, orc_obs, pts[17].copy(), 1.06, flags=0)
    assert 17 in res.idx and res.nearest_idx == 17 and res.nearest_dist == 0.0
    # capacity 0 and below the count: the full count, only the first neighbours and their edges
    q = np.array([0.5, 0.5, 0.0, 3.0])
    full = _full_check(t, orc, pts, P, orc_obs, q, 4.0, flags=0)
    assert full.count > 10
    for cap in (0, 5):
        res = _full_check(t, orc, pts, P, orc_obs, q, 4.0, flags=0, capacity=cap)
        assert res.count == full.count and len(res.idx) == cap and len(res.edge_dist) == 2 * cap
        assert set(res.idx.tolist()) <= set(full.idx.tolist())
    # a root-only tree, and a tree whose nodes all sit in the unsorted tail
    tr, orr = _tree(ctx, ROOT[None, :])
    _full_check(tr, orr, ROOT[None, :], P, orc_obs, np.array([0.3, -0.2, 0.0, 5.9]), 2.0)
    tail_pts = _samples(33, 500)
    tt, ot = _tree(ctx)
    for p in tail_pts:
        tt.insert(p)
        ot.insert(p)
    for k in range(5):
        _full_check(tt, ot, tail_pts, P, orc_obs, _samples(34 + k, 1)[0], 6.0, delta=4.0)
    # rows that outgrow the scratch: every node of a 600-pose tree, in a fresh result (grown, then the call repeats)
    # and in the tree's own scratch (grown by the first call, reused by the second)
    big = _samples(40, 600)
    tb, ob = _tree(ctx, big)
    for k in range(2):
        qk = np.array([0.0, 0.0, 0.0, 1.0 + k])
        res = _full_check(tb, ob, big, P, orc_obs, qk, float("inf"), flags=0)
        assert res.trajectories.sizes()[1] > 16384
        own = extend_query_dubins(tb, P, qk, float("inf"), RHO, R_TURN)
        (ga, ea), (gb, eb) = _order(own), _order(res)
        assert np.array_equal(own.idx[ga], res.idx[gb])
        assert np.array_equal(_bits(own.edge_dist[ea]), _bits(res.edge_dist[eb]))
        assert np.array_equal(own.edge_collide[ea], res.edge_collide[eb])
    # inactive polygons, RRTQX_CHECK_IGNORE_ACTIVE, and an empty polygon set
    obstacles = W.c4_city_blocks()
    active = (np.arange(len(obstacles)) % 3 != 0).astype(np.uint8)
    Pi = PolygonSet(ctx)
    Pi.upload(obstacles, active=active)
    q = np.array([0.5, 0.5, 0.0, 3.0])
    a = _full_check(t, orc, pts, Pi, orc_obs, q, 6.0, flags=0, active=active)
    b = _full_check(t, orc, pts, Pi, orc_obs, q, 6.0, flags=A.CHECK_IGNORE_ACTIVE)
    assert a.count > 10 and np.any(a.edge_collide != b.edge_collide)
    P0 = PolygonSet(ctx)
    P0.upload([])
    res = _full_check(t, orc, pts, P0, [], q, 4.0, flags=0)
    assert not res.edge_collide.any()


def test_refusals(ctx):
    P = PolygonSet(ctx)
    P.upload(W.c4_city_blocks()[:5])
    q = np.array([0.0, 0.0, 0.0, 1.0])
    bad = [DeviceTree(ctx, 3, wraps=(2,), wrap_points=(TWO_PI,)),
           DeviceTree(ctx, 4, wraps=(2, 3), wrap_points=(TWO_PI, TWO_PI)),
           DeviceTree(ctx, 4, wraps=(0,), wrap_points=(TWO_PI,)),
           DeviceTree(ctx, 4, wraps=(3,), wrap_points=(2 * 3.14159,)),
           DeviceTree(ctx, 4)]
    for t in bad:
        t.insert_batch(_samples(50, 100)[:, :t.d])
        with pytest.raises(A.RRTQXError) as e:
            extend_query_dubins(t, P, q, 1.0, RHO, R_TURN)
        assert e.value.status == A.ERR_UNSUPPORTED
    t, _ = _tree(ctx)
    with pytest.raises(A.RRTQXError) as e:
        extend_query_dubins(t, P, q, 1.0, RHO, R_TURN)
    assert e.value.status == A.ERR_EMPTY_TREE
    t.insert_batch(_samples(51, 100))
    S = SphereSet(ctx, np.zeros((1, 3)), np.ones(1))
    with pytest.raises(A.RRTQXError) as e:   # the SimpleEdge call still refuses the Dubins tree
        extend_query(t, S, q, 1.0, RHO)
    assert e.value.status == A.ERR_UNSUPPORTED
