"""The CPU oracle's wrap-around kd tree equals the brute-force ghost model of tests/wrap_model.py: range sets and
keys bit for bit, nearest node and distance bits, on every wrap configuration of the GPU wrap tests (one to four
wrap dimensions, wraps on grid axes and off them) with points and queries on the seams.  This is what lets
test_gpu_wrap.py compare the device with the oracle and mean more than "device equals port"."""
import numpy as np
import pytest

import oracle
import wrap_model as M


def _oracle(cfg, pts):
    d, wraps, wps, _ = cfg
    orc = oracle.KDTree(d, wraps, wps)
    orc.insert_batch(pts)
    return orc


@pytest.mark.parametrize("name", list(M.CONFIGS))
def test_oracle_range_and_nearest_equal_the_model(name):
    cfg = M.CONFIGS[name]
    d, wraps, wps, _ = cfg
    pts = M.points(1, 3000, cfg)
    qs = M.queries(2, 150, cfg, pts)
    orc = _oracle(cfg, pts)
    for r in M.radii(wps):
        for qi, q in enumerate(qs):
            oi, ok = orc.find_within_range(r, q)
            orc.empty(oi)
            mi, mk = M.range_query(pts, q, r, wraps, wps)
            o = np.argsort(oi, kind="stable")
            assert np.array_equal(oi[o], mi), (name, r, qi)
            assert np.array_equal(ok[o].view(np.uint64), mk.view(np.uint64)), (name, r, qi)
    oi, od = orc.nearest_batch(qs)
    for qi, q in enumerate(qs):
        mi, md = M.nearest(pts, q, wraps, wps)
        assert od[qi].view(np.uint64) == np.float64(md).view(np.uint64), (name, qi)
        assert oi[qi] == mi, (name, qi)


@pytest.mark.parametrize("name", [n for n, c in M.CONFIGS.items() if len(c[1]) >= 2])
def test_identity_order_decides_keys_at_large_radii(name):
    """At 1.3 P some nodes are reached by two identities at different distances, so the key depends on which
    identity comes first: the configurations really exercise the ghost order and the dedup."""
    cfg = M.CONFIGS[name]
    d, wraps, wps, _ = cfg
    pts = M.points(1, 3000, cfg)
    r = M.radii(wps)[-1]
    differing = 0
    for q in M.queries(2, 150, cfg, pts)[:40]:
        seen = {}
        for ident in [q] + list(M.ghosts(q, wraps, wps, lambda: r)):
            dist = M.euclid(ident, pts)
            for v in np.nonzero(dist < r)[0][:200]:
                if v in seen and seen[v] != dist[v]:
                    differing += 1
                seen.setdefault(v, dist[v])
    assert differing > 0


@pytest.mark.parametrize("name", list(M.CONFIGS))
def test_nearest_tie_across_identities_keeps_the_real_one(name):
    """A (wrap coordinate 0) and B (wrap coordinate P) sit at the same distance from a query at 0: the real
    identity reaches A, the ghost reaches B.  B is inserted first, so "smallest index" would pick it; strict <
    across identities keeps A."""
    cfg = M.CONFIGS[name]
    pts, q, a = M.tie_tree(cfg)
    orc = _oracle(cfg, pts)
    i, dist = orc.find_nearest(q)
    mi, md = M.nearest(pts, q, cfg[1], cfg[2])
    assert i == mi == a
    assert np.float64(dist).view(np.uint64) == np.float64(md).view(np.uint64)

