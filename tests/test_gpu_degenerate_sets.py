"""GPU parity on degenerate point sets: a pile of 300 identical points and scattered pairs, integer lattices (d = 2,
3, 4) with radii on lattice distances and the root at exactly r, flat and collinear sets, far finite outliers, NaN /
+inf / -inf nodes, an extent that overflows, and a NaN root (tests/nearest_model.py).

Every set runs through every query path: the v5 range kernel with a uniform radius and with per-query radii, the
two-pass range kernel, nearest with one thread per query (>= 4096 queries), one warp per query (forced, and small
batches), and the extend query on a sample.  Range: index sets and keys bit for bit against the CPU oracle.
Nearest: distances bit for bit (NaN as NaN) and the node of the device's documented rule (minimum radicand, then
smallest index; a NaN radicand to the root answers the root), which test_nearest_model.py pins to the oracle."""
import ctypes as C
import os
from contextlib import contextmanager

import numpy as np
import pytest

import nearest_model as M
import oracle
from rrtqx_3d_b200 import _abi as A
from rrtqx_3d_b200 import workloads as W
from rrtqx_3d_b200.device import DeviceTree, SphereSet, extend_query
from test_gpu_wrap import _gpu, _orc, _same

pytestmark = pytest.mark.gpu

RADIUS_MENU = (0.5, 1.0, 3.0, 0.0, -1.0, np.nan, 1e-300)    # per-query radii, relative to the set's radius


@contextmanager
def _env(ctx, name):
    """A diagnostic switch of the library (read at context creation and reload) for the duration of a with-block."""
    os.environ[name] = "1"
    ctx.reload_tuning()
    try:
        yield
    finally:
        del os.environ[name]
        ctx.reload_tuning()


def _model_nearest(pts, qs):
    out = [M.nearest(pts, q) for q in qs]
    return np.array([o[0] for o in out]), np.array([o[1] for o in out]), [o[2] for o in out]


def _same_nearest(gi, gd, mi, md, what):
    nan = np.isnan(md)
    assert np.array_equal(np.isnan(gd), nan), f"{what}: NaN distances differ"
    bad = np.nonzero(gd[~nan].view(np.uint64) != md[~nan].view(np.uint64))[0]
    assert len(bad) == 0, f"{what}: distance of query {np.nonzero(~nan)[0][bad[0]]} differs"
    bad = np.nonzero(gi != mi)[0]
    assert len(bad) == 0, f"{what}: query {bad[0]} -> node {gi[bad[0]]}, the rule gives {mi[bad[0]]}"


def _trees(ctx, pts):
    d = pts.shape[1]
    orc = oracle.KDTree(d)
    orc.insert_batch(pts)
    t = DeviceTree(ctx, d)
    t.insert_batch(pts)
    return orc, t


@pytest.mark.parametrize("name", M.SETS)
def test_range_every_path(ctx, name):
    pts, qs, r, _ = M.point_set(name)
    orc, t = _trees(ctx, pts)
    for rr in M.radii_for(name, r):
        want = _orc(orc, qs, rr)
        _same(_gpu(t, qs, rr), want, f"{name} r = {rr!r}")
        with _env(ctx, "RRTQX_RANGE_TWO_PASS"):
            _same(_gpu(t, qs, rr), want, f"{name} r = {rr!r}, two-pass")
    radii = np.ascontiguousarray(np.array(RADIUS_MENU)[np.arange(len(qs)) % len(RADIUS_MENU)] * r)
    radii[7] = np.inf                                   # one list of every node
    want = _orc(orc, qs, ranges=radii)
    _same(_gpu(t, qs, None, ranges=radii), want, f"{name} per-query radii")
    with _env(ctx, "RRTQX_RANGE_TWO_PASS"):
        _same(_gpu(t, qs, None, ranges=radii), want, f"{name} per-query radii, two-pass")


@pytest.mark.parametrize("name", M.SETS)
def test_nearest_every_path(ctx, name):
    pts, qs, _, case = M.point_set(name)
    orc, t = _trees(ctx, pts)
    mi, md, ties = _model_nearest(pts, qs)
    oi, od = orc.nearest_batch(qs, nthreads=8)
    assert np.array_equal(np.isnan(od), np.isnan(md))
    assert all(oi[k] in ties[k] for k in range(len(qs))), f"{name}: the oracle's node is outside the tie set"
    assert len(qs) >= 4096
    gi, gd = t.nearest(qs)                              # one thread per query
    _same_nearest(gi, gd, mi, md, f"{name} thread per query")
    with _env(ctx, "RRTQX_NEAREST_WARP"):
        gi, gd = t.nearest(qs)
    _same_nearest(gi, gd, mi, md, f"{name} warp per query")
    n_front = _n_front(qs)
    for lo, hi in ((0, 1), (n_front - 3, n_front), (200, n_front)):   # small batches take the warp kernel
        gi, gd = t.nearest(np.ascontiguousarray(qs[lo:hi]))
        _same_nearest(gi, gd, mi[lo:hi], md[lo:hi], f"{name} queries {lo}:{hi}")
    if case is not None:
        q, want = case
        gi, gd = t.nearest(np.tile(q, (4096, 1)))
        assert np.all(gi == want), f"{name}: the node across the cell boundary was pruned"


def _n_front(qs):
    """Rows in front of the uniform queries: nodes, special placements, then NaN, inf and 1e200 (the last)."""
    return int(np.flatnonzero(np.all(qs == 1e200, axis=1))[0]) + 1


@pytest.mark.parametrize("name", M.SETS)
def test_extend_query(ctx, building2, name):
    """Nearest (the model's rule), range (oracle), node check (explicitNodeCheck with the quick pass) and, at d = 3,
    the edge flags of every neighbour against the oracle; at d != 3 the edge flags are 0."""
    pts, qs, r, _ = M.point_set(name)
    d = pts.shape[1]
    orc, t = _trees(ctx, pts)
    centers, sradii, _ = building2
    S = SphereSet(ctx, centers, sradii)
    sph, ns = oracle.make_spheres(centers, sradii)
    L = oracle.lib()
    P = lambda a: oracle._p(np.ascontiguousarray(a, dtype=np.float64), oracle.c_f64p)
    rr = M.radii_for(name, r)[-1]
    for qi in list(range(0, 200, 25)) + list(range(200, _n_front(qs))):   # some nodes, every special placement
        p = qs[qi]
        res = extend_query(t, S, p, rr, W.ROBOT_RADIUS, A.CHECK_QUICK_PASS, capacity=1 << 14)
        mi, md, _ = M.nearest(pts, p)
        assert res.nearest_idx == mi, (name, qi, res.nearest_idx, mi)
        assert (np.isnan(md) and np.isnan(res.nearest_dist)) or res.nearest_dist == md, (name, qi)
        p3 = np.r_[p, np.zeros(3)][:3]
        c = C.c_double()
        hit = L.orc_point_check(sph, ns, 0, P(p3), W.ROBOT_RADIUS, C.byref(c))
        assert (res.point_collides, np.float64(res.point_cert).view(np.uint64)) == (bool(hit), np.float64(c.value).view(np.uint64)), (name, qi)
        oi, ok = orc.find_within_range(rr, p)
        orc.empty(oi)
        assert res.count == len(oi), (name, qi)
        go, oo = np.argsort(res.idx), np.argsort(oi)
        assert np.array_equal(res.idx[go], oi[oo]), (name, qi)
        assert np.array_equal(res.dist[go].view(np.uint64), ok[oo].view(np.uint64)), (name, qi)
        if d != 3:
            assert not res.fwd.any() and not res.rev.any()
            continue
        for k in range(res.count):
            nb = pts[res.idx[k]]
            assert res.fwd[k] == L.orc_edge_check_all(sph, ns, 0, P(p), P(nb), W.ROBOT_RADIUS, 0), (name, qi, k)
            assert res.rev[k] == L.orc_edge_check_all(sph, ns, 0, P(nb), P(p), W.ROBOT_RADIUS, 0), (name, qi, k)
