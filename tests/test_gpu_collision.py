"""GPU parity: edge / node collision checks and the obstacle sweeps vs the oracle.
Collision booleans must be bit-exact (same IEEE operations, same order)."""
import ctypes as C

import numpy as np
import pytest

import oracle
from rrtqx_3d_b200 import _abi as A
from rrtqx_3d_b200 import workloads as W
from rrtqx_3d_b200.device import (DeviceTree, EdgeSet, SphereSet, edge_check_batch, node_check_batch,
                                   segment_check_batch)

pytestmark = pytest.mark.gpu


def _orc_edges(sph, ns, pts, src, dst, rho, fma=0):
    out = np.zeros(len(src), dtype=np.uint8)
    pts = np.ascontiguousarray(pts)
    oracle.lib().orc_edge_check_batch(sph, ns, oracle._p(pts, oracle.c_f64p), 3, oracle._p(src, oracle.c_i32p),
                                      oracle._p(dst, oracle.c_i32p), 0, len(src), rho, fma,
                                      oracle._p(out, oracle.c_u8p), 4)
    return out


def test_edge_check_building2(ctx, building2):
    centers, radii, _ = building2
    pts, _, _ = W.c2_workload(20000, 1)
    n_e = 200000
    u = W.splitmix64(77, 0, 2 * n_e)
    src = (u[:n_e] % np.uint64(len(pts))).astype(np.int32)
    # mostly short edges (neighbours in index space are not neighbours in space: mix both)
    dst = (u[n_e:] % np.uint64(len(pts))).astype(np.int32)
    dst[::5] = src[::5]                      # zero-length edges: collide with every active obstacle (DRRT_Q.jl:1208)
    active = np.ones(len(radii), dtype=np.uint8)
    active[::7] = 0
    sph, ns = oracle.make_spheres(centers, radii, unused=1 - active)
    t = DeviceTree(ctx, 3)
    t.insert_batch(pts)
    S = SphereSet(ctx, centers, radii, active)
    for fma in (0, 1):
        got = edge_check_batch(t, S, src, dst, W.ROBOT_RADIUS, flags=A.CHECK_FMA_DOT if fma else 0)
        want = _orc_edges(sph, ns, pts, src, dst, W.ROBOT_RADIUS, fma)
        assert np.array_equal(got, want)
        assert got[::5].all()
    # every obstacle forced active
    sph_all, _ = oracle.make_spheres(centers, radii)
    got = edge_check_batch(t, S, src, dst, W.ROBOT_RADIUS, flags=A.CHECK_IGNORE_ACTIVE)
    assert np.array_equal(got, _orc_edges(sph_all, ns, pts, src, dst, W.ROBOT_RADIUS))
    # no active obstacle: nothing collides, not even zero-length edges
    S.update(0, active=np.zeros(len(radii), dtype=np.uint8))
    assert not edge_check_batch(t, S, src, dst, W.ROBOT_RADIUS).any()


def test_segment_check_short_edges_near_surfaces(ctx, building2):
    # segments placed around the obstacle surfaces so that many land within ulps of the threshold
    centers, radii, _ = building2
    n = 100000
    base = W.uniform_points(31, n, [-1.0] * 3, [1.0] * 3)
    base /= np.linalg.norm(base, axis=1, keepdims=True)
    k = np.arange(n) % len(radii)
    scale = (radii[k] + W.ROBOT_RADIUS) * (1.0 + (W.uniform01(32, 0, n) - 0.5) * 0.02)
    starts = centers[k] + base * scale[:, None]
    ends = starts + W.uniform_points(33, n, [-0.5] * 3, [0.5] * 3)
    sph, ns = oracle.make_spheres(centers, radii)
    S = SphereSet(ctx, centers, radii)
    got = segment_check_batch(ctx, S, starts, ends, W.ROBOT_RADIUS)
    L = oracle.lib()
    want = np.array([L.orc_edge_check_all(sph, ns, 0, oracle._p(np.ascontiguousarray(starts[i]), oracle.c_f64p),
                                          oracle._p(np.ascontiguousarray(ends[i]), oracle.c_f64p), W.ROBOT_RADIUS, 0)
                     for i in range(0, n, 10)], dtype=np.uint8)
    assert np.array_equal(got[::10], want)
    assert 0.2 < got.mean() < 0.8


def test_node_check_both_variants(ctx, building2):
    centers, radii, _ = building2
    pts = W.uniform_points(41, 50000, [-20.0] * 3, [20.0] * 3)
    active = np.ones(len(radii), dtype=np.uint8)
    active[3] = 0
    sph, ns = oracle.make_spheres(centers, radii, unused=1 - active)
    S = SphereSet(ctx, centers, radii, active)
    L = oracle.lib()
    for flags, fn in ((A.CHECK_QUICK_PASS, L.orc_point_check), (0, L.orc_point_check_3d)):
        got, cert = node_check_batch(ctx, S, pts, W.ROBOT_RADIUS, flags)
        want = np.zeros(len(pts), dtype=np.uint8)
        wcert = np.zeros(len(pts))
        c = C.c_double(0.0)
        for i in range(len(pts)):
            want[i] = fn(sph, ns, 0, oracle._p(np.ascontiguousarray(pts[i]), oracle.c_f64p), W.ROBOT_RADIUS, C.byref(c))
            wcert[i] = c.value
        assert np.array_equal(got, want)
        assert np.array_equal(cert.view(np.uint64), wcert.view(np.uint64))


def _neighbour_graph(ctx, pts, r):
    """All ordered pairs within r (the RRTx neighbour graph) + a parent per node."""
    t = DeviceTree(ctx, 3)
    t.insert_batch(pts)
    res, total = t.range_query(pts, r, want_dist=False)
    counts, offsets = res.layout()
    idx, _ = res.fetch(want_dist=False)
    src = np.empty(total, dtype=np.int32)
    for q in range(len(pts)):
        src[offsets[q]:offsets[q] + counts[q]] = q
    keep = src != idx
    src, dst = src[keep], idx[keep]
    parent = np.arange(len(pts), dtype=np.int32) - 1    # chain parents; node 0 has none
    return t, src, dst, parent


def test_obstacle_add_and_remove_sweep(ctx):
    pts, _, _ = W.c2_workload(20000, 1)
    t, src, dst, parent = _neighbour_graph(ctx, pts, 2.0)
    centers, radii = W.c3_obstacles(12)
    S = SphereSet(ctx, centers, radii)
    E = EdgeSet(t)
    E.upload(src, dst, parent)
    ob_ids = np.arange(len(radii), dtype=np.int32)
    res = E.add_sweep(S, ob_ids, W.ROBOT_RADIUS, W.DELTA, flags=A.SWEEP_STATS)   # node-centric kernel + statistics
    ge, gn = res.fetch()
    n_eh, n_nh, n_cand, n_tests = res.sizes()
    fast = E.add_sweep(S, ob_ids, W.ROBOT_RADIUS, W.DELTA)                         # edge-centric kernel (default)
    fe, fn = fast.fetch()
    assert np.array_equal(fe, ge) and np.array_equal(fn, gn) and fast.sizes()[2:] == (-1, -1)

    # oracle: CSR in edge-id order per start node
    orc = oracle.KDTree(3)
    orc.insert_batch(pts)
    order = np.argsort(src, kind="stable")
    row_ptr = np.zeros(len(pts) + 1, dtype=np.int64)
    np.add.at(row_ptr, src + 1, 1)
    row_ptr = np.cumsum(row_ptr)
    col = np.ascontiguousarray(dst[order])
    eid = order.astype(np.int32)
    L = oracle.lib()
    blocked, orphans = set(), set()
    tot_cand = tot_tests = 0
    sph, _ = oracle.make_spheres(centers, radii)
    cap = len(src) + 8
    be = np.zeros(cap, dtype=np.int32)
    on = np.zeros(len(pts) + 8, dtype=np.int32)
    for o in range(len(radii)):
        nb, no, nc, nt = C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_int64(0)
        rc = L.orc_obstacle_add_sweep(orc.h, C.byref(sph[o]), W.ROBOT_RADIUS, W.DELTA, oracle._p(row_ptr, oracle.c_i64p),
                                      oracle._p(col, oracle.c_i32p), oracle._p(parent, oracle.c_i32p), 0,
                                      oracle._p(be, oracle.c_i32p), C.byref(nb), cap, oracle._p(on, oracle.c_i32p),
                                      C.byref(no), len(on), C.byref(nc), C.byref(nt))
        assert rc == 0
        blocked.update(eid[be[:nb.value]].tolist())
        orphans.update(on[:no.value].tolist())
        tot_cand += nc.value
        tot_tests += nt.value
    assert set(ge.tolist()) == blocked and len(ge) == len(blocked) == n_eh
    assert set(gn.tolist()) == orphans and len(gn) == n_nh
    assert (n_cand, n_tests) == (tot_cand, tot_tests)
    assert len(blocked) > 100 and len(orphans) > 10

    # remove obstacle 0 (Otte semantics: still active while tested): blocked edges that hit
    # obstacle 0 and no other obstacle are restored
    inf = np.zeros(len(src), dtype=np.uint8)
    inf[ge] = 1
    others = np.arange(1, len(radii), dtype=np.int32)
    rr = E.remove_sweep(S, 0, others, inf, W.ROBOT_RADIUS, W.DELTA)
    re_, rn_ = rr.fetch()
    inf_csr = np.ascontiguousarray(inf[order])
    oth, n_oth = oracle.make_spheres(centers[1:], radii[1:])
    nr, nq = C.c_int64(0), C.c_int64(0)
    rc = L.orc_obstacle_remove_sweep(orc.h, C.byref(sph[0]), 1, oth, n_oth, W.ROBOT_RADIUS, W.DELTA,
                                     oracle._p(row_ptr, oracle.c_i64p), oracle._p(col, oracle.c_i32p),
                                     oracle._p(inf_csr, oracle.c_u8p), 0, oracle._p(be, oracle.c_i32p), C.byref(nr), cap,
                                     oracle._p(on, oracle.c_i32p), C.byref(nq), len(on))
    assert rc == 0
    assert set(re_.tolist()) == set(eid[be[:nr.value]].tolist())
    assert set(rn_.tolist()) == set(on[:nq.value].tolist())
    assert nr.value > 0
    # QX semantics (obstacle disabled before the loop, DRRT_Q.jl:3301-3302): nothing restored
    rq = E.remove_sweep(S, 0, others, inf, W.ROBOT_RADIUS, W.DELTA, flags=A.SWEEP_REMOVED_INACTIVE)
    assert rq.sizes()[0] == 0 and rq.sizes()[1] == 0


def _orc_obstacles_2d(polyset):
    obs = []
    for i in range(len(polyset.kind)):
        ob = oracle.Obstacle2D()
        ob.kind = int(polyset.kind[i])
        ob.pos[0], ob.pos[1] = polyset.centers[i]
        ob.radius = polyset.radii[i]
        ob.life_span = float("inf")
        ob.unused = 0
        if ob.kind == 3:
            v = np.ascontiguousarray(polyset.verts[polyset.vptr[i]:polyset.vptr[i + 1]])
            ob.n_vert = len(v)
            ob._keep = v
            ob.poly = oracle._p(v, oracle.c_f64p)
        obs.append(ob)
    return obs


def test_polygon_world_segment_and_dubins_checks(ctx):
    """DRRT.jl:1523-1578 + DRRT_DubinsEdge_functions.jl:750-774 against the oracle, bit-exact booleans."""
    from rrtqx_3d_b200.device import PolygonSet, dubins_edge_check_batch, segment_check_2d_batch
    obstacles = W.c4_city_blocks()[:40]
    obstacles += [("ball", (5.0, 5.0), 2.0), ("ball", (-20.0, 31.0), 4.0),
                  ("polygon", np.array([[0.0, 0.0], [3.0, 0.5], [1.0, 4.0]])),          # triangle
                  ("polygon", np.array([[30.0, 30.0], [30.0, 36.0]]))]                   # degenerate 2-vertex polygon
    P = PolygonSet(ctx)
    P.upload(obstacles)
    orc = _orc_obstacles_2d(P)
    L = oracle.lib()
    f = lambda a: oracle._p(np.ascontiguousarray(a, dtype=np.float64), oracle.c_f64p)
    n = 20000
    starts = W.uniform_points(61, n, [-50.0, -50.0], [50.0, 50.0])
    ends = starts + W.uniform_points(62, n, [-4.0, -4.0], [4.0, 4.0])
    ends[::9, 0] = starts[::9, 0]                  # exactly vertical segments (the 1e-6 branch of segmentDistSqrd)
    ends[::11] = starts[::11]                      # zero-length segments
    rad = 0.5
    got = segment_check_2d_batch(P, starts, ends, rad)
    want = np.zeros(n, dtype=np.uint8)
    import ctypes as C
    for i in range(n):
        for ob in orc:
            if L.orc_edge_check_2d(C.byref(ob), f(starts[i]), f(ends[i]), rad):
                want[i] = 1
                break
    assert np.array_equal(got, want) and 0.05 < want.mean() < 0.9
    # Dubins edges with arc-line-arc trajectories
    nodes, s3, e3, ptr, traj = W.c4_workload(5000, 3000)
    got = dubins_edge_check_batch(P, s3[:, :2], e3[:, :2], ptr, traj, 0.5, 1.0)
    want = np.zeros(len(s3), dtype=np.uint8)
    for i in range(len(s3)):
        t = np.ascontiguousarray(traj[ptr[i]:ptr[i + 1]])
        for ob in orc:
            if L.orc_edge_check_dubins(C.byref(ob), f(s3[i, :2]), f(e3[i, :2]), f(t), len(t), 0.5, 1.0):
                want[i] = 1
                break
    assert np.array_equal(got, want) and 0.05 < want.mean() < 0.95
    # inactive obstacles are skipped
    P.upload(obstacles, active=np.zeros(len(obstacles)))
    assert not segment_check_2d_batch(P, starts, ends, rad).any()


def test_edge_check_grid_path_pathological_obstacles(ctx, building2):
    """Large batches bin the obstacles into a grid; obstacles the reference collides with everything
    (NaN centre -> !(NaN > thr)) or with huge radii must still be met by every edge."""
    centers, radii, _ = building2
    pts, _, _ = W.c2_workload(30000, 1)
    n_e = 50000
    u = W.splitmix64(78, 0, 2 * n_e)
    src = (u[:n_e] % np.uint64(len(pts))).astype(np.int32)
    dst = ((u[:n_e] + u[n_e:] % np.uint64(50)) % np.uint64(len(pts))).astype(np.int32)
    t = DeviceTree(ctx, 3)
    t.insert_batch(pts)
    for variant in ("nan_centre", "inf_radius", "far_outlier", "single_cell"):
        c, r = centers.copy(), radii.copy()
        if variant == "nan_centre":
            c[5, 1] = np.nan
        elif variant == "inf_radius":
            r[7] = np.inf
        elif variant == "far_outlier":
            c[3] = [1e6, -1e6, 1e6]
        else:
            c[:] = c[0]                       # all obstacles at one point: degenerate grid extents
        S = SphereSet(ctx, c, r)
        sph, ns = oracle.make_spheres(c, r)
        got = edge_check_batch(t, S, src, dst, W.ROBOT_RADIUS)
        want = _orc_edges(sph, ns, pts, src, dst, W.ROBOT_RADIUS)
        assert np.array_equal(got, want), variant
        if variant in ("nan_centre", "inf_radius"):
            assert got.all()


def test_resident_edge_set_grows_with_the_planner(ctx):
    """Neighbour-graph residency (rrtqx_edges_append / rrtqx_edges_set_parents): a graph grown in stages --
    new nodes inserted into the tree, their edges appended, parents re-pointed -- gives the same sweep results
    as one upload of the final graph (which the test above pins to the oracle)."""
    pts, _, _ = W.c2_workload(12000, 1)
    t_full, src, dst, parent = _neighbour_graph(ctx, pts, 2.2)
    centers, radii = W.c3_obstacles(10)
    S = SphereSet(ctx, centers, radii)
    ob_ids = np.arange(len(radii), dtype=np.int32)
    E_full = EdgeSet(t_full)
    E_full.upload(src, dst, parent)
    want_e, want_n = E_full.add_sweep(S, ob_ids, W.ROBOT_RADIUS, W.DELTA).fetch()

    # staged: nodes [0, n1) with the edges among them, then two more stages
    t = DeviceTree(ctx, 3)
    E = EdgeSet(t)
    stages = [4000, 9000, 12000]
    eid_map = []                                   # staged edge id -> full edge id
    prev = 0
    for k, n_k in enumerate(stages):
        t.insert_batch(pts[prev:n_k])
        hi = np.maximum(src, dst)
        sel = np.nonzero((hi >= prev) & (hi < n_k))[0]   # edges whose later endpoint arrives in this stage
        par_k = np.where(parent[:n_k] < n_k, parent[:n_k], -1).astype(np.int32)
        if k == 0:
            E.upload(src[sel], dst[sel], par_k)
        else:
            E.append(src[sel], dst[sel])
            changed = np.arange(n_k, dtype=np.int32)     # re-point everything (idempotent for unchanged nodes)
            E.set_parents(changed, par_k)
        eid_map.append(sel)
        prev = n_k
        if k == 1:   # a sweep in the middle of the growth also works (CSR rebuilt lazily)
            mid = E.add_sweep(S, ob_ids, W.ROBOT_RADIUS, W.DELTA)
            assert mid.sizes()[0] > 0
    eid_map = np.concatenate(eid_map)
    assert len(E) == len(src)
    got_e, got_n = E.add_sweep(S, ob_ids, W.ROBOT_RADIUS, W.DELTA).fetch()
    assert np.array_equal(np.sort(eid_map[got_e]), want_e)
    # parents that point to a later node were masked to -1 only while that node did not exist; at the end the
    # parent arrays agree, so the orphan sets agree
    assert np.array_equal(got_n, want_n)
    # the statistics kernel (node-centric, uses the CSR + lmax of the rebuilt set) agrees as well
    st = E.add_sweep(S, ob_ids, W.ROBOT_RADIUS, W.DELTA, flags=A.SWEEP_STATS)
    se, sn = st.fetch()
    assert np.array_equal(se, got_e) and np.array_equal(sn, got_n)


def test_edge_check_cover_lists_short_edges(ctx):
    """Very large batches of SHORT edges take the two-stage kernels with cover lists (csrc/collide_queue.cuh; forced
    here at test size): one
    fine-grid cell list per edge instead of the coarse rows.  Mixed with long, zero-length and out-of-box edges,
    against obstacle sets that keep the cover (C3-style), overflow its budget (huge spheres: coarse rows), are
    tiny compared with the box, or sit outside the tree's box; booleans bit-exact, with and without the FMA dot."""
    pts, _, _ = W.c2_workload(30000, 1)
    t, src, dst, _ = _neighbour_graph(ctx, pts, 1.3)
    assert len(src) > 100000
    src, dst = src.copy(), dst.copy()
    dst[5::101] = (src[5::101] + 7777) % len(pts)            # long edges (coarse rows)
    dst[::97] = src[::97]                                    # zero-length edges
    far = np.array([[1e3, 1e3, 1e3], [1e3 + 0.2, 1e3, 1e3 + 0.1], [-500.0, 3.0, 2.0], [-500.1, 3.2, 2.0]])
    n0 = len(pts)
    pts2 = np.ascontiguousarray(np.vstack([pts, far]))       # short edges far outside the obstacle box
    t2 = DeviceTree(ctx, 3)
    t2.insert_batch(pts2)
    src = np.concatenate([src, np.array([n0, n0 + 1, n0 + 2, n0 + 3], dtype=np.int32)])
    dst = np.concatenate([dst, np.array([n0 + 1, n0, n0 + 3, n0 + 2], dtype=np.int32)])
    rng = np.random.default_rng(5)
    sets = {
        "c3": W.c3_obstacles(256),
        "huge": (rng.uniform(-20, 20, (3000, 3)), rng.uniform(10.0, 15.0, 3000)),        # cover over budget
        "tiny": (rng.uniform(-20, 20, (2000, 3)), rng.uniform(0.01, 0.2, 2000)),
        "mixed": (np.vstack([rng.uniform(-20, 20, (60, 3)), [[1e3, 1e3, 1e3]], [[np.nan, 0.0, 0.0]]]),
                  np.concatenate([rng.uniform(0.5, 3.0, 60), [1.0], [1.0]])),
    }
    import os
    os.environ["RRTQX_COVER_MIN_ITEMS"] = "1"   # the two-stage path is the default only above ~2e6 edges
    ctx.reload_tuning()                         # switches are read at context creation / on request only
    try:
        for name, (c, r) in sets.items():
            c, r = np.ascontiguousarray(c, dtype=np.float64), np.ascontiguousarray(r, dtype=np.float64)
            S = SphereSet(ctx, c, r)
            sph, ns = oracle.make_spheres(c, r)
            for fma in (0, 1):
                got = edge_check_batch(t2, S, src, dst, W.ROBOT_RADIUS, flags=A.CHECK_FMA_DOT if fma else 0)
                want = _orc_edges(sph, ns, pts2, src, dst, W.ROBOT_RADIUS, fma)
                assert np.array_equal(got, want), (name, fma, int((got != want).sum()))
            assert got[:len(got) - 4:97].all()
            if name in ("c3", "tiny"):
                assert 0 < got.sum() < len(got)
    finally:
        del os.environ["RRTQX_COVER_MIN_ITEMS"]
        ctx.reload_tuning()


def test_two_stage_and_thread_per_edge_paths_agree(ctx):
    """The same edge batch and add sweep through the library's own choice (the thread-per-item kernel over the obstacle grid at
    this size; the two-stage kernels take over above ~1e6 items), the thread-per-edge kernels forced
    (RRTQX_EDGE_NO_QUEUE=1) and the two-stage kernels forced (RRTQX_COVER_MIN_ITEMS=1): identical flags / id lists, and equal to the oracle."""
    import os
    pts, _, _ = W.c2_workload(12000, 1)
    t, src, dst, parent = _neighbour_graph(ctx, pts, 1.6)
    centers, radii = W.c3_obstacles(64)
    S = SphereSet(ctx, centers, radii)
    sph, ns = oracle.make_spheres(centers, radii)
    E = EdgeSet(t)
    E.upload(src, dst, parent)
    ids = np.arange(len(radii), dtype=np.int32)
    small = slice(0, 6000)                      # 4096 <= n < 16384: thread-per-item kernel over the obstacle grid by default
    want = _orc_edges(sph, ns, pts, src, dst, W.ROBOT_RADIUS)
    results = {}
    # the add sweep over a resident edge set takes the obstacle-centric item grid by default; RRTQX_NO_ITEM_GRID=1 gives
    # the edge-centric kernels, whose own variants are then selected as before
    for mode, env in (("default", {}), ("edge_centric", {"RRTQX_NO_ITEM_GRID": "1"}),
                      ("no_queue", {"RRTQX_NO_ITEM_GRID": "1", "RRTQX_EDGE_NO_QUEUE": "1"}),
                      ("forced", {"RRTQX_NO_ITEM_GRID": "1", "RRTQX_COVER_MIN_ITEMS": "1"})):
        for k, v in env.items():
            os.environ[k] = v
        ctx.reload_tuning()
        try:
            full = edge_check_batch(t, S, src, dst, W.ROBOT_RADIUS)
            part = edge_check_batch(t, S, src[small], dst[small], W.ROBOT_RADIUS)
            sw = E.add_sweep(S, ids, W.ROBOT_RADIUS, W.DELTA)
            results[mode] = (full, part, *sw.fetch())
        finally:
            for k in env:
                del os.environ[k]
            ctx.reload_tuning()
    for mode, (full, part, be, on) in results.items():
        assert np.array_equal(full, want), mode
        assert np.array_equal(part, want[small]), mode
        assert np.array_equal(be, results["default"][2]) and np.array_equal(on, results["default"][3]), mode
    assert 0 < want.sum() < len(want) and len(results["default"][2]) > 0


def test_bad_edge_endpoints_fail_the_call_host_and_device_arrays(ctx, building2):
    """An out-of-range endpoint must give RRTQX_ERR_INVALID -- also when src / dst live on the device, where the
    host cannot look at them (validated inside the gathering kernels / by a small kernel at edge upload)."""
    import torch
    centers, radii, _ = building2
    pts, _, _ = W.c2_workload(6000, 1)
    t = DeviceTree(ctx, 3)
    t.insert_batch(pts)
    S = SphereSet(ctx, centers, radii)
    src = np.arange(5000, dtype=np.int32)
    dst = src[::-1].copy()
    good = edge_check_batch(t, S, src, dst, W.ROBOT_RADIUS)
    for bad_value in (-1, 6000, 2 ** 31 - 1):
        for n_e in (100, 5000):           # tiled kernel / thread-per-item kernel over the obstacle grid
            s2, d2 = src[:n_e].copy(), dst[:n_e].copy()
            d2[n_e // 2] = bad_value
            with pytest.raises(A.RRTQXError) as ei:
                edge_check_batch(t, S, s2, d2, W.ROBOT_RADIUS)
            assert ei.value.status == A.ERR_INVALID
            ds, dd = torch.from_numpy(s2).cuda(), torch.from_numpy(d2).cuda()
            out = torch.zeros(n_e, dtype=torch.uint8, device="cuda")
            with pytest.raises(A.RRTQXError) as ei:
                edge_check_batch(t, S, ds.data_ptr(), dd.data_ptr(), W.ROBOT_RADIUS, n_edges=n_e, out=out.data_ptr())
            assert ei.value.status == A.ERR_INVALID
        E = EdgeSet(t)
        d2 = dst.copy()
        d2[17] = bad_value
        ds, dd = torch.from_numpy(src).cuda(), torch.from_numpy(d2).cuda()
        with pytest.raises(A.RRTQXError):
            E.upload(ds.data_ptr(), dd.data_ptr(), None, n_edges=len(src))
    # the context is still healthy afterwards
    assert np.array_equal(edge_check_batch(t, S, src, dst, W.ROBOT_RADIUS), good)


def test_cached_obstacle_tables_follow_updates(ctx):
    """The active-obstacle table / obstacle grid / cover lists are cached per obstacle-set content: an in-place
    update, another robot radius, another flag or another obstacle set must never see stale tables."""
    pts, _, _ = W.c2_workload(12000, 1)
    t = DeviceTree(ctx, 3)
    t.insert_batch(pts)
    u = W.splitmix64(5, 0, 2 * 20000)
    src = (u[:20000] % np.uint64(len(pts))).astype(np.int32)
    dst = ((src.astype(np.int64) + 1 + (u[20000:] % np.uint64(40)).astype(np.int64)) % len(pts)).astype(np.int32)
    c, r = W.c3_obstacles(64)
    S = SphereSet(ctx, c, r)
    c2, r2 = c[::-1].copy() * 0.5, r[::-1].copy()
    S2 = SphereSet(ctx, c2, r2)
    import os
    for forced in (False, True):
        if forced:
            os.environ["RRTQX_COVER_MIN_ITEMS"] = "1"
        ctx.reload_tuning()
        try:
            act = np.ones(64, np.uint8)
            S.update(0, radii=r, active=act)
            for step in range(4):
                sph, ns = oracle.make_spheres(c, r, unused=1 - act)
                for rho in (W.ROBOT_RADIUS, 1.25):
                    for _ in range(2):      # second call: served from the cache
                        assert np.array_equal(edge_check_batch(t, S, src, dst, rho), _orc_edges(sph, ns, pts, src, dst, rho))
                sph_all, _ = oracle.make_spheres(c, r)
                assert np.array_equal(edge_check_batch(t, S, src, dst, W.ROBOT_RADIUS, flags=A.CHECK_IGNORE_ACTIVE),
                                      _orc_edges(sph_all, ns, pts, src, dst, W.ROBOT_RADIUS))
                sph2, ns2 = oracle.make_spheres(c2, r2)
                assert np.array_equal(edge_check_batch(t, S2, src, dst, W.ROBOT_RADIUS), _orc_edges(sph2, ns2, pts, src, dst, W.ROBOT_RADIUS))
                act[step * 16:(step + 1) * 16:2] = 0
                r = r.copy()
                r[step] += 0.75
                S.update(0, radii=r, active=act)
        finally:
            os.environ.pop("RRTQX_COVER_MIN_ITEMS", None)
            ctx.reload_tuning()


def test_contexts_come_and_go():
    """Several contexts in one process, created and destroyed in turn: the per-context scratch (obstacle tables,
    cover lists, pair lists) and the per-context shared-memory opt-in of the range kernel live and die with their
    context (a recycled address must never meet another context's buffers)."""
    from rrtqx_3d_b200.device import Context
    pts, qs, r = W.c2_workload(20000, 3000)
    c, rad = W.c3_obstacles(32)
    sph, ns = oracle.make_spheres(c, rad)
    src = np.arange(10000, dtype=np.int32)
    dst = (src + 7) % 20000
    want = _orc_edges(sph, ns, pts, src, dst, W.ROBOT_RADIUS)
    orc = oracle.KDTree(3)
    orc.insert_batch(pts)
    oc, _, _, _ = orc.range_batch(r, qs, want_lists=False, nthreads=8)
    alive = []
    for round_ in range(4):
        cx = Context(0)
        t = DeviceTree(cx, 3)
        t.insert_batch(pts)
        S = SphereSet(cx, c, rad)
        assert np.array_equal(edge_check_batch(t, S, src, dst, W.ROBOT_RADIUS), want)
        res, _ = t.range_query(qs, r)
        counts, _ = res.layout()
        assert np.array_equal(counts, oc)
        if round_ % 2 == 0:
            alive.append((cx, t, S, res))      # keep two contexts alive next to the following ones
        else:
            res.close(); S.close(); t.close(); cx.close()
    for cx, t, S, res in alive:
        assert np.array_equal(edge_check_batch(t, S, src, dst, W.ROBOT_RADIUS), want)
        res.close(); S.close(); t.close(); cx.close()


def test_handles_may_be_destroyed_in_any_order():
    """Garbage-collected hosts (Julia finalizers, Python __del__ of objects in reference cycles) destroy handles in
    arbitrary order: the context before its trees, a tree before its edge set and results.  Nothing may crash or
    leave a CUDA error behind for the next call."""
    from rrtqx_3d_b200.device import Context, EdgeSet
    pts, qs, r = W.c2_workload(5000, 100)
    c, rad = W.c3_obstacles(16)
    src = np.arange(4000, dtype=np.int32)
    dst = (src + 3) % 5000
    for order in ("ctx_first", "tree_first"):
        cx = Context(0)
        t = DeviceTree(cx, 3)
        t.insert_batch(pts)
        S = SphereSet(cx, c, rad)
        E = EdgeSet(t)
        E.upload(src, dst, None)
        res, _ = t.range_query(qs, r)
        sw = E.add_sweep(S, np.arange(16, dtype=np.int32), W.ROBOT_RADIUS, W.DELTA)
        if order == "ctx_first":
            cx.close(); sw.close(); E.close(); res.close(); S.close(); t.close()
        else:
            t.close(); E.close(); res.close(); sw.close(); cx.close(); S.close()
        cx.close(); t.close()          # a second destroy of a dead handle is a no-op
        # a fresh context right afterwards sees no stale error
        c2 = Context(0)
        t2 = DeviceTree(c2, 3)
        t2.insert_batch(pts)
        S2 = SphereSet(c2, c, rad)
        assert edge_check_batch(t2, S2, src, dst, W.ROBOT_RADIUS).shape == (4000,)
        S2.close(); t2.close(); c2.close()


def test_resident_edge_check_equals_batch_check_and_oracle(ctx):
    """rrtqx_edges_check_batch (every resident out-edge, prepared per-item records: FP32 midpoint / half-length for the
    collect stage, exact end points for the test stage) gives the flags of rrtqx_edge_check_batch and of the oracle;
    zero-length edges, long edges, edges far outside the obstacle box, pathological obstacle sets, both dot forms,
    and an edge set that grows and gets new parents in between."""
    import os
    pts, _, _ = W.c2_workload(12000, 1)
    t, src, dst, parent = _neighbour_graph(ctx, pts, 1.6)
    n0 = len(pts)
    far = np.array([[900.0, 900.0, 900.0], [900.2, 900.1, 900.0], [-700.0, 3.0, 2.0], [-700.1, 3.1, 2.2]])
    pts2 = np.ascontiguousarray(np.vstack([pts, far]))
    t.insert_batch(far)
    extra_s = np.array([n0, n0 + 1, n0 + 2, n0 + 3, 5, 17, 40, 41], dtype=np.int32)
    extra_d = np.array([n0 + 1, n0, n0 + 3, n0 + 2, 5, 9000, 40, n0], dtype=np.int32)   # incl. zero-length and long edges
    src2, dst2 = np.concatenate([src, extra_s]), np.concatenate([dst, extra_d])
    rng = np.random.default_rng(8)
    sets = {
        "c3": W.c3_obstacles(256),
        "huge": (rng.uniform(-20, 20, (3000, 3)), rng.uniform(10.0, 15.0, 3000)),        # cover over budget
        "tiny": (rng.uniform(-20, 20, (2000, 3)), rng.uniform(0.01, 0.2, 2000)),
        "mixed": (np.vstack([rng.uniform(-20, 20, (60, 3)), [[1e3, 1e3, 1e3]], [[np.nan, 0.0, 0.0]]]),
                  np.concatenate([rng.uniform(0.5, 3.0, 60), [1.0], [1.0]])),
    }
    E = EdgeSet(t)
    E.upload(src, dst, np.concatenate([parent, np.full(len(far), -1, dtype=np.int32)]))
    E.append(extra_s, extra_d)                       # the records follow the grown edge set
    for name, (c, r) in sets.items():
        c, r = np.ascontiguousarray(c, dtype=np.float64), np.ascontiguousarray(r, dtype=np.float64)
        S = SphereSet(ctx, c, r)
        sph, ns = oracle.make_spheres(c, r)
        for fma in (0, 1):
            fl = A.CHECK_FMA_DOT if fma else 0
            got = E.check_all(S, W.ROBOT_RADIUS, flags=fl)
            want = _orc_edges(sph, ns, pts2, src2, dst2, W.ROBOT_RADIUS, fma)
            assert np.array_equal(got, want), (name, fma, int((got != want).sum()))
            assert np.array_equal(got, edge_check_batch(t, S, src2, dst2, W.ROBOT_RADIUS, flags=fl)), (name, fma)
        if name in ("c3", "tiny"):
            assert 0 < got.sum() < len(got)
    # the sweep over the same records: forced two-stage path == thread-per-edge path == (already oracle-checked) default
    c, r = sets["c3"]
    S = SphereSet(ctx, c, r)
    ids = np.arange(64, dtype=np.int32)
    ref = E.add_sweep(S, ids, W.ROBOT_RADIUS, W.DELTA).fetch()                  # obstacle-centric item grid
    sph, ns = oracle.make_spheres(c[:64], r[:64])
    for env in ({"RRTQX_NO_ITEM_GRID": "1"}, {"RRTQX_NO_ITEM_GRID": "1", "RRTQX_COVER_MIN_ITEMS": "1"}):
        os.environ.update(env)
        ctx.reload_tuning()
        try:
            other = E.add_sweep(S, ids, W.ROBOT_RADIUS, W.DELTA).fetch()
            flags_ec = E.check_all(S, W.ROBOT_RADIUS)                              # edge-centric resident check
        finally:
            for k in env:
                del os.environ[k]
            ctx.reload_tuning()
        assert np.array_equal(ref[0], other[0]) and np.array_equal(ref[1], other[1]) and len(ref[0]) > 0
        assert np.array_equal(flags_ec, E.check_all(S, W.ROBOT_RADIUS))
    # single obstacles (the planner's real call): a few cells of the grid instead of every item
    for o in (0, 7, 63):
        one = E.add_sweep(S, [o], W.ROBOT_RADIUS, W.DELTA).fetch()
        os.environ["RRTQX_NO_ITEM_GRID"] = "1"
        ctx.reload_tuning()
        try:
            want = E.add_sweep(S, [o], W.ROBOT_RADIUS, W.DELTA).fetch()
        finally:
            del os.environ["RRTQX_NO_ITEM_GRID"]
            ctx.reload_tuning()
        assert np.array_equal(one[0], want[0]) and np.array_equal(one[1], want[1])


@pytest.mark.gpu
def test_sweep_result_is_reusable_and_its_flag_view_matches_the_lists(ctx):
    """The flag compaction cleans the flag arrays behind itself and rrtqx_sweep_result_flags rebuilds the byte view from
    the id lists: one result object reused across sweeps (different obstacle subsets, flag view read in between, a
    larger edge set afterwards) must give what fresh result objects give."""
    from rrtqx_3d_b200.device import SweepResult
    pts, _, _ = W.c2_workload(20000, 1)
    t, src, dst, parent = _neighbour_graph(ctx, pts, 2.0)
    centers, radii = W.c3_obstacles(12)
    S = SphereSet(ctx, centers, radii)
    E = EdgeSet(t)
    E.upload(src, dst, parent)
    reused = SweepResult(ctx)
    for ids in ([0], [3, 4, 5], list(range(12)), [7], [], [1]):
        ids = np.asarray(ids, dtype=np.int32)
        fresh = E.add_sweep(S, ids, W.ROBOT_RADIUS, W.DELTA)
        fe, fn = fresh.fetch()
        E.add_sweep(S, ids, W.ROBOT_RADIUS, W.DELTA, result=reused)
        ge, gn = reused.fetch()
        assert np.array_equal(ge, fe) and np.array_equal(gn, fn)
        assert np.all(np.diff(ge) > 0) and np.all(np.diff(gn) > 0)          # ascending id lists
        for _ in range(2):                                                     # the view can be read repeatedly
            ef, nf = reused.flags(len(src), len(pts))
            assert np.array_equal(np.flatnonzero(ef), ge) and np.array_equal(np.flatnonzero(nf), gn)
            assert set(np.unique(ef)) <= {0, 1} and set(np.unique(nf)) <= {0, 1}
    # remove sweep through the same object, then a LARGER edge set (flag arrays grow: new allocation, zeroed)
    first = E.add_sweep(S, np.arange(12, dtype=np.int32), W.ROBOT_RADIUS, W.DELTA)
    inf = np.zeros(len(src), dtype=np.uint8)
    inf[first.fetch()[0]] = 1
    others = np.arange(1, 12, dtype=np.int32)
    want = E.remove_sweep(S, 0, others, inf, W.ROBOT_RADIUS, W.DELTA).fetch()
    got = E.remove_sweep(S, 0, others, inf, W.ROBOT_RADIUS, W.DELTA, result=reused).fetch()
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    t2, src2, dst2, parent2 = _neighbour_graph(ctx, pts, 2.3)
    assert len(src2) > len(src)
    E2 = EdgeSet(t2)
    E2.upload(src2, dst2, parent2)
    w2 = E2.add_sweep(S, np.arange(12, dtype=np.int32), W.ROBOT_RADIUS, W.DELTA).fetch()
    g2 = E2.add_sweep(S, np.arange(12, dtype=np.int32), W.ROBOT_RADIUS, W.DELTA, result=reused).fetch()
    assert np.array_equal(g2[0], w2[0]) and np.array_equal(g2[1], w2[1])
