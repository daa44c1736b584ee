"""Config C1 replay: the planner's per-iteration geometric work (nearest -> node check -> range(r(n)) ->
2k edge checks -> insert) through the fused rrtqx_extend_query, every iteration compared with the oracle."""
import ctypes as C

import numpy as np
import pytest

import nearest_model as NM
import oracle
from rrtqx_3d_b200 import _abi as A
from rrtqx_3d_b200 import workloads as W
from rrtqx_3d_b200.device import DeviceTree, SphereSet, extend_query

pytestmark = pytest.mark.gpu


def test_c1_replay_matches_oracle(ctx, building2):
    centers, radii, _ = building2
    sph, ns = oracle.make_spheres(centers, radii)          # all 31 spheres forced active (SURVEY 8d C1)
    S = SphereSet(ctx, centers, radii)
    L = oracle.lib()
    P = lambda a: oracle._p(np.ascontiguousarray(a, dtype=np.float64), oracle.c_f64p)
    n_iter = 20000                                          # the full C1 configuration (SURVEY 8d)
    samples = W.uniform_points(1, n_iter, [-W.ENV_RAD] * 3, [W.ENV_RAD] * 3)
    t = DeviceTree(ctx, 3)
    orc = oracle.KDTree(3)
    goal = np.array([4.0, 16.5, -7.5])                      # root of the search tree (experimentsForRRTQX.jl:41)
    t.insert(goal)
    orc.insert(goal)
    bufs = None
    accepted = 0
    for it in range(n_iter):
        p = samples[it]
        n = len(orc)
        r = W.shrinking_ball_radius(n, 3, W.DELTA, W.BALL_CONSTANT)      # rrtqx.jl:382, n = treeSize before the insert
        res = extend_query(t, S, p, r, W.ROBOT_RADIUS, A.CHECK_QUICK_PASS, capacity=4096)
        oi, od = orc.find_nearest(p)
        assert (res.nearest_idx, res.nearest_dist) == (oi, od)
        c = C.c_double()
        hit = L.orc_point_check(sph, ns, 0, P(p), W.ROBOT_RADIUS, C.byref(c))
        assert (res.point_collides, res.point_cert) == (bool(hit), c.value)
        idx, key = orc.find_within_range(r, p)
        orc.empty(idx)
        assert res.count == len(idx)
        go, oo = np.argsort(res.idx), np.argsort(idx)
        assert np.array_equal(res.idx[go], idx[oo])
        assert np.array_equal(res.dist[go].view(np.uint64), key[oo].view(np.uint64))
        if it % 25 == 0 or it < 50:        # edge flags: forward new->n and reverse n->new (not symmetric)
            pts = orc_positions(orc)
            for k in range(len(res.idx)):
                nb = pts[res.idx[k]]
                assert res.fwd[k] == L.orc_edge_check_all(sph, ns, 0, P(p), P(nb), W.ROBOT_RADIUS, 0)
                assert res.rev[k] == L.orc_edge_check_all(sph, ns, 0, P(nb), P(p), W.ROBOT_RADIUS, 0)
        if not res.point_collides:         # the planner only inserts collision-free samples (rrtqx.jl:940-950)
            assert t.insert(p) == orc.insert(p)
            accepted += 1
    assert accepted > 0.6 * n_iter and len(t) == accepted + 1
    # kd topology after thousands of single inserts + re-indexing is still the sequential one
    for a, b in zip(t.kd_fields(), orc.fields()):
        assert np.array_equal(a, b)


def orc_positions(orc):
    n = len(orc)
    ptr = oracle.lib().orc_kd_positions
    ptr.restype = C.POINTER(C.c_double)
    ptr.argtypes = [C.c_void_p]
    return np.ctypeslib.as_array(ptr(orc.h), shape=(n, orc.d))


def test_extend_query_capacity_and_empty_ball(ctx, building2):
    centers, radii, _ = building2
    S = SphereSet(ctx, centers, radii)
    pts, _, _ = W.c2_workload(5000, 1)
    t = DeviceTree(ctx, 3)
    t.insert_batch(pts)
    orc = oracle.KDTree(3)
    orc.insert_batch(pts)
    q = np.array([1.0, 2.0, 3.0])
    res = extend_query(t, S, q, 6.0, 0.5, 0, capacity=16)            # more neighbours than capacity
    idx, _ = orc.find_within_range(6.0, q)
    orc.empty(idx)
    assert res.count == len(idx) > 16 and len(res.idx) == 16 and set(res.idx.tolist()) <= set(idx.tolist())
    res = extend_query(t, S, np.array([500.0, 0.0, 0.0]), 1.0, 0.5, 0)   # empty ball: nearest by brute force
    oi, od = orc.find_nearest(np.array([500.0, 0.0, 0.0]))
    assert res.count == 0 and (res.nearest_idx, res.nearest_dist) == (oi, od)


def test_extend_query_ignores_inactive_entries_of_a_long_obstacle_list(ctx, building2):
    """The reference's obstacle list only grows (expired agent obstacles stay in it, rrtqx.jl:462-530): 5000 entries
    of which 31 are active must work (the kernel's table holds the ACTIVE ones), and the answer must follow an
    in-place update of the flags."""
    centers, radii, _ = building2
    rng = np.random.default_rng(3)
    n_dead = 5000
    allc = np.vstack([rng.uniform(-20, 20, (n_dead, 3)), centers])
    allr = np.concatenate([rng.uniform(1.0, 3.0, n_dead), radii])
    active = np.concatenate([np.zeros(n_dead, np.uint8), np.ones(len(radii), np.uint8)])
    S_long = SphereSet(ctx, allc, allr, active)
    S_ref = SphereSet(ctx, centers, radii)
    pts, _, _ = W.c2_workload(5000, 1)
    t = DeviceTree(ctx, 3)
    t.insert_batch(pts)
    for q in (np.array([1.0, 2.0, 3.0]), np.array([-5.0, 5.0, 0.5]), centers[4] + 0.1):
        a = extend_query(t, S_long, q, 4.0, 0.5, A.CHECK_QUICK_PASS)
        b = extend_query(t, S_ref, q, 4.0, 0.5, A.CHECK_QUICK_PASS)
        assert (a.point_collides, a.point_cert, a.count) == (b.point_collides, b.point_cert, b.count)
        oa, ob = np.argsort(a.idx), np.argsort(b.idx)
        assert np.array_equal(a.idx[oa], b.idx[ob])
        assert np.array_equal(a.fwd[oa], b.fwd[ob]) and np.array_equal(a.rev[oa], b.rev[ob])
    # switch every active obstacle off: nothing collides any more
    S_long.update(n_dead, active=np.zeros(len(radii), np.uint8))
    a = extend_query(t, S_long, centers[4] + 0.1, 4.0, 0.5, A.CHECK_QUICK_PASS)
    assert not a.point_collides and not a.fwd.any() and not a.rev.any()
    # more than 768 ACTIVE obstacles is refused loudly, not silently truncated
    S_big = SphereSet(ctx, allc[:1000], allr[:1000])
    with pytest.raises(A.RRTQXError):
        extend_query(t, S_big, np.array([1.0, 2.0, 3.0]), 4.0, 0.5, 0)


# ------------------------------------------------------------------------ every input of one extend query
_P = lambda a: oracle._p(np.ascontiguousarray(a, dtype=np.float64), oracle.c_f64p)


def _check_extend(t, S, sph, ns, pts, orc, p, r, rho, flags, capacity, count_differ=False):
    """One extend query against the oracle: nearest by the model's rule (nearest_model.py), the neighbour list and
    keys, the node check of the variant `flags` selects, and the edge flags of every neighbour (0 at d != 3).
    With count_differ, returns the number of edges whose flags differ between the two oracle dot-product variants."""
    L = oracle.lib()
    d = pts.shape[1]
    res = extend_query(t, S, p, r, rho, flags, capacity=capacity)
    mi, md, _ = NM.nearest(pts, p)
    assert res.nearest_idx == mi and (np.isnan(md) and np.isnan(res.nearest_dist) or res.nearest_dist == md), \
        (p, r, res.nearest_idx, res.nearest_dist, mi, md)
    c = C.c_double()
    check = L.orc_point_check if flags & A.CHECK_QUICK_PASS else L.orc_point_check_3d
    hit = check(sph, ns, 0, _P(np.r_[p, np.zeros(3)][:3]), rho, C.byref(c))
    assert res.point_collides == bool(hit), (p, flags)
    assert np.float64(res.point_cert).view(np.uint64) == np.float64(c.value).view(np.uint64), (p, flags)
    oi, ok = orc.find_within_range(r, p)
    orc.empty(oi)
    assert res.count == len(oi), (p, r)
    assert len(res.idx) == min(len(oi), capacity)
    if capacity < len(oi):
        assert set(res.idx.tolist()) <= set(oi.tolist())
        return 0
    go, oo = np.argsort(res.idx), np.argsort(oi)
    assert np.array_equal(res.idx[go], oi[oo]), (p, r)
    assert np.array_equal(res.dist[go].view(np.uint64), ok[oo].view(np.uint64)), (p, r)
    if d != 3:
        assert not res.fwd.any() and not res.rev.any()
        return 0
    fma = 1 if flags & A.CHECK_FMA_DOT else 0
    differ = 0
    for k in range(res.count):
        nb = pts[res.idx[k]]
        for got, a, b in ((res.fwd[k], p, nb), (res.rev[k], nb, p)):
            want = L.orc_edge_check_all(sph, ns, 0, _P(a), _P(b), rho, fma)
            assert got == want, (p, k, fma)
            if count_differ:
                differ += want != L.orc_edge_check_all(sph, ns, 0, _P(a), _P(b), rho, 1 - fma)
    return differ


@pytest.mark.parametrize("n", [40, 3000])
@pytest.mark.parametrize("d", [2, 3, 4])
def test_extend_query_every_input(ctx, building2, d, n):
    """d = 2, 3, 4; a tree of 40 nodes (no grid: tail path only) and of 3000; both node checks, both dot products;
    radii r, 0, -1, NaN, +inf, 1e-300 and the root at exactly r; samples equal to nodes, NaN and 1e200 samples;
    zero obstacles; capacity 0."""
    centers, radii, _ = building2
    rng = np.random.default_rng(11 + d)
    pts = rng.uniform(-20.0, 20.0, (n, d))
    pts[0, :] = np.round(pts[0, :])                       # root on integers: root + (3, 4) is exactly r = 5 away
    t = DeviceTree(ctx, d)
    t.insert_batch(pts)
    orc = oracle.KDTree(d)
    orc.insert_batch(pts)
    r = 5.0
    off = np.zeros(d)
    off[:2] = [3.0, 4.0]
    samples = list(rng.uniform(-20.0, 20.0, (6, d))) + [pts[0], pts[1], pts[n // 2], pts[0] + off, pts[0] - off,
                                                       np.full(d, np.nan), np.r_[1.0, np.nan, np.zeros(d - 2)],
                                                       np.full(d, 1e200), np.r_[np.inf, np.zeros(d - 1)]]
    sets = [(SphereSet(ctx, centers, radii), oracle.make_spheres(centers, radii)),
            (SphereSet(ctx), oracle.make_spheres(np.zeros((0, 3)), np.zeros(0)))]
    for S, (sph, ns) in sets:
        for flags in (0, A.CHECK_QUICK_PASS, A.CHECK_FMA_DOT):
            for p in samples:
                for rr in (r, 0.0, -1.0, np.nan, np.inf, 1e-300):
                    _check_extend(t, S, sph, ns, pts, orc, p, rr, W.ROBOT_RADIUS, flags, n + 1)
        for p in samples[:8]:
            _check_extend(t, S, sph, ns, pts, orc, p, r, W.ROBOT_RADIUS, 0, 0)          # capacity 0
    res = extend_query(t, sets[1][0], samples[0], r, W.ROBOT_RADIUS, 0)
    assert not res.point_collides and res.point_cert == np.inf       # no obstacle: certificate +inf


def test_extend_query_root_at_exactly_r(ctx, building2):
    """The root is admitted with <=, every other node with <: on an integer lattice the root at exactly r = 5 is a
    neighbour, the lattice nodes at exactly 5 are not."""
    centers, radii, _ = building2
    pts, _, _, _ = NM.point_set("lattice3")
    t = DeviceTree(ctx, 3)
    t.insert_batch(pts)
    orc = oracle.KDTree(3)
    orc.insert_batch(pts)
    S = SphereSet(ctx, centers, radii)
    sph, ns = oracle.make_spheres(centers, radii)
    for off in ([3.0, 4.0, 0.0], [0.0, -4.0, 3.0], [5.0, 0.0, 0.0]):
        p = pts[0] + np.array(off)
        res = extend_query(t, S, p, 5.0, W.ROBOT_RADIUS, A.CHECK_QUICK_PASS)
        assert 0 in res.idx.tolist() and res.dist[res.idx.tolist().index(0)] == 5.0
        assert np.count_nonzero(res.dist == 5.0) == 1
        _check_extend(t, S, sph, ns, pts, orc, p, 5.0, W.ROBOT_RADIUS, A.CHECK_QUICK_PASS, 4096)


def test_extend_node_check_variants(ctx):
    """explicitNodeCheck with the quick pass (:1520) and without (explicitPointCheck3D, :1558) differ only for NaN
    samples and, at robot radius 0, for a sample exactly on a sphere surface: both cases, both variants."""
    c5, r5 = np.zeros((1, 3)), np.array([5.0])          # building2 covers (3, 4, 0): one sphere alone
    S = SphereSet(ctx, c5, r5)
    sph, ns = oracle.make_spheres(c5, r5)
    L = oracle.lib()
    pts = np.random.default_rng(4).uniform(-20.0, 20.0, (500, 3))
    t = DeviceTree(ctx, 3)
    t.insert_batch(pts)
    orc = oracle.KDTree(3)
    orc.insert_batch(pts)
    cases = [(np.array([3.0, 4.0, 0.0]), 0.0), (np.array([np.nan, 1.0, 2.0]), 0.5), (np.array([np.nan, 1.0, 2.0]), 0.0)]
    for p, rho in cases:
        c = C.c_double()
        assert L.orc_point_check(sph, ns, 0, _P(p), rho, C.byref(c)) != L.orc_point_check_3d(sph, ns, 0, _P(p), rho, C.byref(c))
        for flags in (0, A.CHECK_QUICK_PASS):
            _check_extend(t, S, sph, ns, pts, orc, p, 4.0, rho, flags, 4096)
    for p in (np.array([3.0, 4.0, 1e-9]), np.array([0.0, 0.0, 5.0 + 1e-12]), pts[7], np.array([-8.0, 2.0, 1.0])):
        for flags in (0, A.CHECK_QUICK_PASS):
            _check_extend(t, S, sph, ns, pts, orc, p, 4.0, 0.0, flags, 4096)


def _fma_sensitive_edges(centers, radii, rho, n_want, seed=21):
    """(sample, node) pairs whose edge flags differ between the plain and the FMA dot product of the reference's
    point-to-segment distance: the sample slides along a line until the segment's distance to a sphere crosses
    robotRadius + radius, then the last ulps around the crossing are searched."""
    L = oracle.lib()
    sph, ns = oracle.make_spheres(centers, radii)
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(2000):
        o = int(rng.integers(len(radii)))
        c, thr = centers[o], rho + radii[o]
        n1 = rng.normal(size=3)
        n1 /= np.linalg.norm(n1)
        n2 = np.cross(n1, rng.normal(size=3))
        n2 /= np.linalg.norm(n2)
        e = c + (thr + 1.0) * n1

        def hit(lam, fma):
            return L.orc_edge_check_sphere(C.byref(sph[o]), _P(c + lam * n2), _P(e), rho, fma)

        lo, hi = 0.0, 50.0
        if not hit(lo, 0) or hit(hi, 0):
            continue
        while True:
            mid = 0.5 * (lo + hi)
            if mid <= lo or mid >= hi:
                break
            lo, hi = (mid, hi) if hit(mid, 0) else (lo, mid)
        lam = lo
        for _ in range(64):
            lam = np.nextafter(lam, -np.inf)
        for _ in range(128):
            s = c + lam * n2
            if any(L.orc_edge_check_all(sph, ns, 0, _P(a), _P(b), rho, 0) !=
                   L.orc_edge_check_all(sph, ns, 0, _P(a), _P(b), rho, 1) for a, b in ((s, e), (e, s))):
                out.append((s, e))
                break
            lam = np.nextafter(lam, np.inf)
        if len(out) == n_want:
            break
    return out


def test_extend_fma_dot_edge_flags(ctx, building2):
    """RRTQX_CHECK_FMA_DOT: the edge flags of every neighbour equal the oracle's FMA variant, on samples whose
    edges to a tree node sit within an ulp of a building2 sphere, where the two variants disagree."""
    centers, radii, _ = building2
    pairs = _fma_sensitive_edges(centers, radii, W.ROBOT_RADIUS, 12)
    assert len(pairs) >= 4
    rng = np.random.default_rng(8)
    pts = np.vstack([rng.uniform(-20.0, 20.0, (3000, 3)), [e for _, e in pairs]])
    t = DeviceTree(ctx, 3)
    t.insert_batch(pts)
    orc = oracle.KDTree(3)
    orc.insert_batch(pts)
    S = SphereSet(ctx, centers, radii)
    sph, ns = oracle.make_spheres(centers, radii)
    differ = 0
    for s, e in pairs:
        r = float(np.linalg.norm(s - e)) + 0.5
        for flags in (A.CHECK_FMA_DOT, A.CHECK_FMA_DOT | A.CHECK_QUICK_PASS, 0):
            differ += _check_extend(t, S, sph, ns, pts, orc, s, r, W.ROBOT_RADIUS, flags, 8192, count_differ=True)
    assert differ > 0
