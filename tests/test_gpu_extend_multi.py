"""rrtqx_extend_query_multi / rrtqx_tree_insert_multi: many independent planning instances in lock-step, one launch
per round for the queries and one for the inserts.  Every instance must see exactly what the single calls give it."""
import ctypes as C

import numpy as np
import pytest

import oracle
from rrtqx_3d_b200 import _abi as A
from rrtqx_3d_b200 import workloads as W
from rrtqx_3d_b200.device import (Context, DeviceTree, SphereSet, extend_query, extend_query_multi,
                                  insert_multi)

pytestmark = pytest.mark.gpu

_P = lambda a: oracle._p(np.ascontiguousarray(a, dtype=np.float64), oracle.c_f64p)
GOAL = np.array([4.0, 16.5, -7.5])


def _orc_positions(orc):
    f = oracle.lib().orc_kd_positions
    f.restype = C.POINTER(C.c_double)
    f.argtypes = [C.c_void_p]
    return np.ctypeslib.as_array(f(orc.h), shape=(len(orc), orc.d))


def _bits(x):
    return np.float64(x).view(np.uint64)


def _entries(res):
    """The neighbour list as a set: (idx, dist bits, fwd, rev) in node order."""
    o = np.argsort(res.idx, kind="stable")
    return list(zip(res.idx[o].tolist(), res.dist[o].view(np.uint64).tolist(), res.fwd[o].tolist(), res.rev[o].tolist()))


def _same(a, b, capacity=None):
    """Multi result a equals single result b bit for bit; with a capacity below the count, a's entries are any
    `capacity` of b's complete list."""
    assert (a.nearest_idx, _bits(a.nearest_dist), a.point_collides, _bits(a.point_cert), a.count) == \
        (b.nearest_idx, _bits(b.nearest_dist), b.point_collides, _bits(b.point_cert), b.count)
    if capacity is not None and capacity < b.count:
        assert len(a.idx) == capacity
        assert set(_entries(a)) <= set(_entries(b))
    else:
        assert _entries(a) == _entries(b)


# ------------------------------------------------------------------------ 1. lock-step replay against the oracle
def test_lockstep_replay_matches_oracle(ctx, building2):
    """8 C1-style instances (seeds 1..8), 3000 lock-step rounds: instances 0-5 share building2, instance 6 has its own
    set with every other sphere inactive, instance 7 an empty set.  Each instance against its own oracle tree."""
    centers, radii, _ = building2
    n_inst, n_iter = 8, 3000
    inactive = (np.arange(len(radii)) % 2).astype(bool)
    S_shared = SphereSet(ctx, centers, radii)
    S6 = SphereSet(ctx, centers, radii, (~inactive).astype(np.uint8))
    S7 = SphereSet(ctx)
    sets = [S_shared] * 6 + [S6, S7]
    osets = [oracle.make_spheres(centers, radii)] * 6 + [oracle.make_spheres(centers, radii, unused=inactive),
                                                        oracle.make_spheres(np.zeros((0, 3)), np.zeros(0))]
    samples = [W.uniform_points(1 + i, n_iter, [-W.ENV_RAD] * 3, [W.ENV_RAD] * 3) for i in range(n_inst)]
    trees = [DeviceTree(ctx, 3) for _ in range(n_inst)]
    orcs = [oracle.KDTree(3) for _ in range(n_inst)]
    assert insert_multi(trees, np.tile(GOAL, (n_inst, 1))).tolist() == [0] * n_inst
    for o in orcs:
        o.insert(GOAL)
    L = oracle.lib()
    for it in range(n_iter):
        pts = np.stack([s[it] for s in samples])
        ranges = [W.shrinking_ball_radius(len(o), 3, W.DELTA, W.BALL_CONSTANT) for o in orcs]
        res = extend_query_multi(trees, sets, pts, ranges, W.ROBOT_RADIUS, A.CHECK_QUICK_PASS, capacity=4096)
        for i, (r, orc, (sph, ns)) in enumerate(zip(res, orcs, osets)):
            p = pts[i]
            assert (r.nearest_idx, r.nearest_dist) == orc.find_nearest(p), (it, i)
            c = C.c_double()
            hit = L.orc_point_check(sph, ns, 0, _P(p), W.ROBOT_RADIUS, C.byref(c))
            assert (r.point_collides, _bits(r.point_cert)) == (bool(hit), _bits(c.value)), (it, i)
            idx, key = orc.find_within_range(ranges[i], p)
            orc.empty(idx)
            assert r.count == len(idx), (it, i)
            go, oo = np.argsort(r.idx), np.argsort(idx)
            assert np.array_equal(r.idx[go], idx[oo]), (it, i)
            assert np.array_equal(r.dist[go].view(np.uint64), key[oo].view(np.uint64)), (it, i)
            if it % 25 == 0 or it < 50:
                opos = _orc_positions(orc)
                for k in range(len(r.idx)):
                    nb = opos[r.idx[k]]
                    assert r.fwd[k] == L.orc_edge_check_all(sph, ns, 0, _P(p), _P(nb), W.ROBOT_RADIUS, 0), (it, i, k)
                    assert r.rev[k] == L.orc_edge_check_all(sph, ns, 0, _P(nb), _P(p), W.ROBOT_RADIUS, 0), (it, i, k)
        acc = [i for i in range(n_inst) if not res[i].point_collides]
        if acc:
            got = insert_multi([trees[i] for i in acc], pts[acc])
            assert got.tolist() == [orcs[i].insert(pts[i]) for i in acc]
    for t, o in zip(trees, orcs):
        assert len(t) == len(o) > 65        # every tree crossed the re-index threshold (64 unsorted nodes)
        for a, b in zip(t.kd_fields(), o.fields()):
            assert np.array_equal(a, b)
    assert len(trees[7]) == n_iter + 1       # no obstacle: every sample accepted


# ------------------------------------------------------------------------ 2. multi equals single, bit for bit
def _twin_trees(ctx, d, rng):
    """Trees of very different sizes, built twice identically: root only, a 40-node tail, 3000 nodes, 10^5 nodes."""
    sets = [rng.uniform(-20.0, 20.0, (n, d)) for n in (1, 40, 3000, 100_000)]
    for pts in sets:
        pts[0, :] = np.round(pts[0, :])
    twins = []
    for pts in sets:
        pair = []
        for _ in range(2):
            t = DeviceTree(ctx, d)
            t.insert_batch(pts)
            pair.append(t)
        twins.append(pair)
    return sets, twins


def _sqdist(a, b):
    s = 0.0
    for c in range(len(a)):
        s = s + (a[c] - b[c]) * (a[c] - b[c])
    return s


@pytest.mark.parametrize("d", [2, 3, 4])
def test_multi_equals_single(ctx, building2, d):
    centers, radii, _ = building2
    rng = np.random.default_rng(40 + d)
    sets, twins = _twin_trees(ctx, d, rng)
    A_trees, B_trees = [p[0] for p in twins], [p[1] for p in twins]
    S = SphereSet(ctx, centers, radii)
    n = len(sets)
    big = sets[3]
    node = big[1234]
    exact = float(np.sqrt(_sqdist(big[0] + 0.37, node)))
    rounds = [  # (points, ranges) per instance
        ([s[min(5, len(s) - 1)] + 0.25 for s in sets], [5.0, 5.0, 2.5, 1.5]),
        ([s[0] + 0.37 for s in sets], [0.0, -1.0, np.nan, np.inf]),
        ([big[0] + 0.37] * n, [3.0, 0.5, exact, np.nextafter(exact, np.inf)]),   # node 1234 at exactly `exact`
        ([np.full(d, np.nan), np.full(d, 1e200), sets[2][17].copy(), node.copy()], [4.0, 4.0, 4.0, 1.0]),
        ([np.r_[1.0, np.nan, np.zeros(d - 2)], np.r_[np.inf, np.zeros(d - 1)], rng.uniform(-20, 20, d),
          rng.uniform(-20, 20, d)], [1e-300, 6.0, 6.0, 6.0]),
    ]
    edge_hits = 0
    for flags in (0, A.CHECK_QUICK_PASS, A.CHECK_FMA_DOT, A.CHECK_FMA_DOT | A.CHECK_QUICK_PASS):
        for pts, ranges in rounds:
            pts = np.stack(pts)
            full = [extend_query(B_trees[i], S, pts[i], ranges[i], W.ROBOT_RADIUS, flags, capacity=200_000)
                    for i in range(n)]
            for cap in (200_000, 0, 7):
                got = extend_query_multi(A_trees, [S] * n, pts, ranges, W.ROBOT_RADIUS, flags, capacity=cap)
                for i in range(n):
                    _same(got[i], full[i], cap)
            edge_hits += sum(int(f.fwd.sum()) + int(f.rev.sum()) for f in full)
    assert (edge_hits > 0) == (d == 3)      # SimpleEdge checks run on 3-D trees only
    # the root-only and 40-node trees are tail-only: no grid index
    assert len(A_trees[0]) == 1 and len(A_trees[1]) == 40


def test_multi_inserts_equal_single_inserts(ctx):
    """insert_multi keeps every tree's kd fields exactly what rrtqx_tree_insert builds."""
    rng = np.random.default_rng(5)
    n, steps = 5, 300
    A_trees = [DeviceTree(ctx, 3) for _ in range(n)]
    B_trees = [DeviceTree(ctx, 3) for _ in range(n)]
    for k in range(steps):
        pts = rng.uniform(-20, 20, (n, 3))
        pick = [i for i in range(n) if (k + i) % 3 != 0 or k == 0]
        got = insert_multi([A_trees[i] for i in pick], pts[pick])
        want = [B_trees[i].insert(pts[i]) for i in pick]
        assert got.tolist() == want
    for a, b in zip(A_trees, B_trees):
        assert len(a) == len(b)
        for x, y in zip(a.kd_fields(), b.kd_fields()):
            assert np.array_equal(x, y)
        assert np.array_equal(a.positions(), b.positions())


# ------------------------------------------------------------------------ 3. interleaving and state
def test_interleaved_single_and_multi_and_sphere_updates(ctx, building2):
    centers, radii, _ = building2
    rng = np.random.default_rng(9)
    n = 6
    trees = []
    for i in range(n):
        t = DeviceTree(ctx, 3)
        t.insert_batch(rng.uniform(-20, 20, (2000, 3)))
        trees.append(t)
    S_toggle = SphereSet(ctx, centers, radii)
    S_fixed = SphereSet(ctx, centers, radii)
    sets = [S_toggle, S_fixed] * (n // 2)
    active = np.ones(len(radii), np.uint8)
    for rnd in range(12):
        pts = rng.uniform(-20, 20, (n, 3))
        ranges = rng.uniform(2.0, 6.0, n)
        multi = extend_query_multi(trees, sets, pts, ranges, W.ROBOT_RADIUS, A.CHECK_QUICK_PASS, capacity=4096)
        single = [extend_query(trees[i], sets[i], pts[i], ranges[i], W.ROBOT_RADIUS, A.CHECK_QUICK_PASS)
                  for i in range(n)]
        for a, b in zip(multi, single):
            _same(a, b)
        again = extend_query_multi(trees, sets, pts, ranges, W.ROBOT_RADIUS, A.CHECK_QUICK_PASS, capacity=4096)
        for a, b in zip(again, single):
            _same(a, b)
        # toggle obstacles of the shared set between rounds: every instance that uses it sees the change
        active[rng.integers(len(radii), size=8)] ^= 1
        S_toggle.update(0, active=active)
        inside = np.stack([centers[(rnd + i) % len(radii)] for i in range(n)])   # samples inside a sphere
        probe = extend_query_multi(trees, sets, inside, np.full(n, 3.0), W.ROBOT_RADIUS, A.CHECK_QUICK_PASS)
        for i in range(n):
            o = (rnd + i) % len(radii)
            ref_active = active if sets[i] is S_toggle else np.ones(len(radii), np.uint8)
            sph, ns = oracle.make_spheres(centers, radii, unused=ref_active == 0)
            c = C.c_double()
            hit = oracle.lib().orc_point_check(sph, ns, 0, _P(inside[i]), W.ROBOT_RADIUS, C.byref(c))
            assert (probe[i].point_collides, _bits(probe[i].point_cert)) == (bool(hit), _bits(c.value)), (rnd, i, o)
        if rnd % 3 == 2:
            insert_multi(trees, rng.uniform(-20, 20, (n, 3)))
    assert any(not a for a in active)


def test_more_instances_than_sms(ctx, building2):
    """N = 300 blocks (more than the 148 SMs): every instance is correct."""
    centers, radii, _ = building2
    rng = np.random.default_rng(300)
    n = 300
    trees = []
    for i in range(n):
        t = DeviceTree(ctx, 3)
        t.insert_batch(rng.uniform(-20, 20, (int(rng.integers(1, 400)), 3)))
        trees.append(t)
    S = SphereSet(ctx, centers, radii)
    for _ in range(3):
        pts = rng.uniform(-20, 20, (n, 3))
        ranges = rng.uniform(1.0, 8.0, n)
        multi = extend_query_multi(trees, [S] * n, pts, ranges, W.ROBOT_RADIUS, A.CHECK_QUICK_PASS)
        for i in range(n):
            _same(multi[i], extend_query(trees[i], S, pts[i], ranges[i], W.ROBOT_RADIUS, A.CHECK_QUICK_PASS))
        insert_multi(trees, pts)


# ------------------------------------------------------------------------ 4. launch counts
def test_steady_state_launch_counts(ctx, building2):
    centers, radii, _ = building2
    rng = np.random.default_rng(4)
    n = 16
    trees = []
    for _ in range(n):
        t = DeviceTree(ctx, 3)
        t.insert_batch(rng.uniform(-20, 20, (3000, 3)))
        t.reindex()
        trees.append(t)
    S = SphereSet(ctx, centers, radii)
    extend_query_multi(trees, [S] * n, rng.uniform(-20, 20, (n, 3)), np.full(n, 4.0), W.ROBOT_RADIUS)   # compaction
    for _ in range(5):
        k0 = ctx.kernel_launches()
        extend_query_multi(trees, [S] * n, rng.uniform(-20, 20, (n, 3)), np.full(n, 4.0), W.ROBOT_RADIUS)
        k1 = ctx.kernel_launches()
        insert_multi(trees, rng.uniform(-20, 20, (n, 3)))
        k2 = ctx.kernel_launches()
        assert (k1 - k0, k2 - k1) == (1, 1)
    L = ctx.L
    k0 = ctx.kernel_launches()
    assert L.rrtqx_extend_query_multi(None, None, 0, None, None, 0.5, 0, 0, *([None] * 9)) == A.OK
    assert L.rrtqx_tree_insert_multi(None, 0, None, None) == A.OK
    assert ctx.kernel_launches() == k0


# ------------------------------------------------------------------------ 5. refusals
def _raw_multi(ctx, trees, sets, pts, ranges, capacity=64):
    """The C call with sentinel-filled outputs; returns (status, message, outputs)."""
    n = len(trees)
    th = (A.vp * n)(*[None if t is None else t.h for t in trees])
    sh = (A.vp * n)(*[None if s is None else s.h for s in sets])
    outs = [np.full(n, -7, np.int32), np.full(n, -7.0), np.full(n, 7, np.uint8), np.full(n, -7.0),
            np.full(n, -7, np.int32), np.full(n * 64, -7, np.int32), np.full(n * 64, -7.0),
            np.full(n * 64, 7, np.uint8), np.full(n * 64, 7, np.uint8)]
    st = ctx.L.rrtqx_extend_query_multi(th, sh, n, A.ptr(pts) if isinstance(pts, np.ndarray) else pts, A.ptr(ranges),
                                        W.ROBOT_RADIUS, 0, capacity, *[A.ptr(o) for o in outs])
    return st, (ctx.L.rrtqx_last_error(ctx.h) or b"").decode(), outs


def _untouched(outs):
    return all(np.all(o == (7 if o.dtype == np.uint8 else -7)) for o in outs)


def test_refusals(ctx, building2):
    centers, radii, _ = building2
    rng = np.random.default_rng(12)

    def tree(d=3, n=500, c=ctx, **kw):
        t = DeviceTree(c, d, **kw)
        if n:
            t.insert_batch(rng.uniform(0.5, 6.0, (n, d)))
        return t

    S = SphereSet(ctx, centers, radii)
    good = [tree(), tree()]
    pts, ranges = rng.uniform(-5, 5, (2, 3)), np.array([3.0, 3.0])

    def ok_after():
        st, msg, outs = _raw_multi(ctx, good, [S, S], pts, ranges)
        assert st == A.OK, msg
        assert not _untouched(outs)
        assert insert_multi(good, rng.uniform(-5, 5, (2, 3))).shape == (2,)

    ctx2 = Context(0)
    other = tree(c=ctx2)
    S_other = SphereSet(ctx2, centers, radii)
    S_big = SphereSet(ctx, rng.uniform(-20, 20, (800, 3)), np.full(800, 0.1))
    wrap = tree(n=500, wraps=[2], wrap_points=[10.0])
    cases = [
        ([good[0], None], [S, S], A.ERR_INVALID, "instance 1"),
        ([good[0], good[1]], [S, None], A.ERR_INVALID, "instance 1"),
        ([good[0], other], [S, S], A.ERR_INVALID, "another context"),
        ([good[0], good[1]], [S, S_other], A.ERR_INVALID, "another context"),
        ([good[0], tree(d=2)], [S, S], A.ERR_INVALID, "dimension"),
        ([good[0], good[0]], [S, S], A.ERR_INVALID, "twice"),
        ([good[0], wrap], [S, S], A.ERR_UNSUPPORTED, "instance 1"),
        ([tree(n=0), good[1]], [S, S], A.ERR_EMPTY_TREE, "instance 0"),
        ([good[0], good[1]], [S, S_big], A.ERR_INVALID, "instance 1"),
    ]
    for trees, sets, status, words in cases:
        st, msg, outs = _raw_multi(ctx, trees, sets, pts, ranges)
        assert st == status and words in msg, (st, msg, words)
        assert _untouched(outs), words
        ok_after()
    st, msg, outs = _raw_multi(ctx, good, [S, S], pts, ranges, capacity=-1)
    assert st == A.ERR_INVALID and "capacity" in msg and _untouched(outs)
    ok_after()
    import torch
    dpts = torch.tensor(pts, device="cuda")
    st, msg, outs = _raw_multi(ctx, good, [S, S], int(dpts.data_ptr()), ranges)
    assert st == A.ERR_INVALID and "host array" in msg and _untouched(outs)
    ok_after()
    # the multi insert: the same handle rules; nothing inserted on refusal
    sizes = [len(t) for t in good]
    for trees, words in (([good[0], None], "NULL"), ([good[0], other], "another context"),
                         ([good[0], tree(d=2)], "dimension"), ([good[1], good[1]], "twice")):
        with pytest.raises(A.RRTQXError, match=words) as e:
            insert_multi(trees, rng.uniform(-5, 5, (2, 3)))
        assert e.value.status == A.ERR_INVALID
        assert [len(t) for t in good] == sizes
        ok_after()
        sizes = [len(t) for t in good]
    th = (A.vp * 2)(good[0].h, good[1].h)
    assert ctx.L.rrtqx_tree_insert_multi(th, 2, int(torch.zeros(6, dtype=torch.float64, device="cuda").data_ptr()),
                                         None) == A.ERR_INVALID
    assert [len(t) for t in good] == sizes
    ok_after()
