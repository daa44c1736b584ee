"""Known answers PRODUCED BY THE REFERENCE (Julia), found in its own tree: R/BVPData/BVPDistFromStaticObs_*.txt.

Each row is [p, min_j euclid(p, c_j) - radius_argmin] over the static spheres of R/environments/buildingsSmall.txt,
written by saveBVPDists (R/DRRT_Q.jl:91-97) from findClosestObs (R/DRRT_Q.jl:127-142); tests/golden/
make_reference_outputs.py collects them (and proves which obstacle file they belong to).  They pin the arithmetic every
part of the path is made of -- the left-to-right radicand and the correctly rounded sqrt of euclidianDist
(R/DRRT_distance_functions.jl) -- through three different routes of the oracle, bit for bit:
kdFindNearest (distance of the winner), kdFindWithinRange (the JList keys) and explicitPointCheck3D (the certificate),
and, with -m gpu, through the same three routes of the CUDA library.  Twelve values do not pin the whole path (the
Julia script of tests/test_reference_vectors.py does that), but they are the reference's own output, not ours."""
import ctypes as C
import json
import math
import os

import numpy as np
import pytest

import oracle

HERE = os.path.dirname(os.path.abspath(__file__))


def _load():
    d = json.load(open(os.path.join(HERE, "golden", "reference_bvp_dists.json")))
    S = np.array([[float.fromhex(x) for x in s] for s in d["spheres_hex"]])
    rows = np.array([[float.fromhex(x) for x in r["v"]] for r in d["rows_hex"]])
    arg = np.array([r["argmin"] for r in d["rows_hex"]])
    return S, rows, arg


def test_fixture_is_the_reference_output():
    """The stored rows are bit patterns copied from the reference's files (make_reference_outputs.py).  What ties them
    to the stored obstacles is what identified the obstacle file: findClosestObs in plain IEEE double arithmetic (first
    minimum wins) reproduces every recorded distance and argmin from the stored spheres, bit for bit."""
    S, rows, arg = _load()
    assert S.shape == (15, 4) and rows.shape == (12, 4)
    for (x, y, z, want), a in zip(rows, arg):
        best, rad, j_best = -1.0, 0.0, -1
        for j, (cx, cy, cz, r) in enumerate(S.tolist()):
            d = math.sqrt((x - cx) ** 2 + (y - cy) ** 2 + (z - cz) ** 2)
            if d < best or best == -1.0:
                best, rad, j_best = d, r, j
        assert j_best == a and (best - rad).hex() == float(want).hex()


def test_oracle_reproduces_the_reference_distances_bit_for_bit():
    S, rows, arg = _load()
    t = oracle.KDTree(3)
    t.insert_batch(S[:, :3])
    L = oracle.lib()
    sph, ns = oracle.make_spheres(S[:, :3], S[:, 3])
    for (x, y, z, want), a in zip(rows, arg):
        q = np.array([x, y, z])
        i, d = t.find_nearest(q)                                   # kdFindNearest: winner and its distance
        assert i == a
        assert d - S[i, 3] == want
        idx, key = t.find_within_range(np.nextafter(d, np.inf), q)  # kdFindWithinRange: JList keys
        t.empty(idx)
        assert a in idx and key[list(idx).index(a)] - S[a, 3] == want
        c = C.c_double(0.0)                                        # explicitPointCheck3D: certificate, robot radius 0
        hit = L.orc_point_check_3d(sph, ns, 0, oracle._p(q, oracle.c_f64p), 0.0, C.byref(c))
        assert hit == (1 if want <= 0.0 else 0)
        if not hit:   # equal radii: the certificate's minimum over (dist - radius) is the recorded value
            assert np.all(S[:, 3] == S[0, 3]) and c.value == want


@pytest.mark.gpu
def test_cuda_path_reproduces_the_reference_distances_bit_for_bit():
    from rrtqx_3d_b200.device import Context, DeviceTree, SphereSet, node_check_batch
    S, rows, arg = _load()
    ctx = Context(0)
    t = DeviceTree(ctx, 3)
    t.insert_batch(S[:, :3])
    q = np.ascontiguousarray(rows[:, :3])
    idx, dist = t.nearest(q)
    assert np.array_equal(idx, arg)
    assert np.array_equal((dist - S[idx, 3]).view(np.uint64), rows[:, 3].copy().view(np.uint64))
    res, total = t.range_query(q, 40.0)        # every centre: keys of all 15 obstacles for all 12 points
    counts, offsets = res.layout()
    ri, rd = res.fetch()
    for k in range(len(q)):
        sl = slice(offsets[k], offsets[k] + counts[k])
        j = list(ri[sl]).index(arg[k])
        assert rd[sl][j] - S[arg[k], 3] == rows[k, 3]
    spheres = SphereSet(ctx, S[:, :3], S[:, 3])
    hit, cert = node_check_batch(ctx, spheres, q, 0.0, 0)
    assert np.all(S[:, 3] == S[0, 3])          # equal radii: the certificate's minimum is the recorded one
    assert np.array_equal(hit, (rows[:, 3] <= 0.0).astype(np.uint8))
    assert np.array_equal(cert[hit == 0].view(np.uint64), rows[hit == 0, 3].copy().view(np.uint64))
