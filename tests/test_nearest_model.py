"""The CPU oracle equals the brute-force model of tests/nearest_model.py on the degenerate point sets: range sets
and keys bit for bit at every test radius, nearest distances bit for bit (NaN as NaN) with the oracle's node inside
the model's tie set.  This is what lets test_gpu_degenerate_sets.py hold the device to the model's tie rule and
mean more than "device equals port"."""
import numpy as np
import pytest

import nearest_model as M
import oracle

N_SAMPLE = 300          # queries per set: the special placements in front, then a stride sample


def _sample(nq):
    return sorted(set(range(260)) | set(range(260, nq, 97)))[:N_SAMPLE]


@pytest.mark.parametrize("name", M.SETS)
def test_oracle_equals_the_model(name):
    pts, qs, r, case = M.point_set(name)
    orc = oracle.KDTree(pts.shape[1])
    orc.insert_batch(pts)
    sample = _sample(len(qs))
    for rr in M.radii_for(name, r):
        for qi in sample:
            oi, ok = orc.find_within_range(rr, qs[qi])
            orc.empty(oi)
            mi, mk = M.range_query(pts, qs[qi], rr)
            o = np.argsort(oi, kind="stable")
            assert np.array_equal(oi[o], mi), (name, rr, qi)
            assert np.array_equal(ok[o].view(np.uint64), mk.view(np.uint64)), (name, rr, qi)
    oi, od = orc.nearest_batch(qs[sample])
    for k, qi in enumerate(sample):
        mi, md, ties = M.nearest(pts, qs[qi])
        assert (np.isnan(od[k]) and np.isnan(md)) or od[k].view(np.uint64) == np.float64(md).view(np.uint64), (name, qi)
        assert oi[k] in ties and mi in ties, (name, qi)
    if case is not None:
        q, want = case
        assert orc.find_nearest(q)[0] == want == M.nearest(pts, q)[0]


def test_the_sets_hold_what_they_are_named_for():
    """Ties and non-finite answers really occur: a test that passes on them proves something."""
    pts, qs, _, _ = M.point_set("lattice3")
    ties = sum(len(M.nearest(pts, q)[2]) > 1 for q in qs[:400])
    assert ties > 20
    idx, key = M.range_query(pts, pts[0] + [3.0, 4.0, 0.0], 5.0)
    assert 0 in idx and key[0] == 5.0                       # the root at exactly r is admitted with <=
    assert not np.any(key[1:] == 5.0)
    pts, qs, _, _ = M.point_set("duplicates")
    assert np.count_nonzero(np.all(pts == [1.25, -3.5, 2.0], axis=1)) == M.PILE
    pts, qs, _, _ = M.point_set("nan_root")
    assert all(M.nearest(pts, q)[:1] == (0,) and np.isnan(M.nearest(pts, q)[1]) for q in qs[:50])
    for name in ("posinf_node", "neginf_node", "overflow_extent"):
        pts, qs, _, (q, want) = M.point_set(name)
        lo, cell, dims = M.grid_dims(pts)
        assert dims[0] == 1 and dims[1] > 8, name          # x has one cell, y a real grid
        cy = [int(np.floor((p[1] - lo[1]) / cell[1])) for p in (q, pts[want], pts[want - 1])]
        assert cy[0] == cy[2] == cy[1] - 1, name            # the nearest is across the boundary, the runner-up is not
