"""Brute-force model of kdFindNearest / kdFindWithinRange on trees without wrap-around, plain numpy float64, and the
degenerate point sets that test_nearest_model.py (model vs CPU oracle) and test_gpu_degenerate_sets.py (model and
oracle vs the device) share.

Radicands are euclidianDist's, in the reference's operation order: ((dx*dx + dy*dy) + dz*dz) + dw*dw, every
operation rounded, no FMA.  Range: the root is admitted with sqrt(s) <= r, every other node with sqrt(s) < r
(kdTree_general.jl:889-919).  Nearest, the device's documented rule: when the radicand to the root is NaN the answer
is the root with that distance (the reference seeds its best distance with the root's, :359-361, and nothing compares
below NaN); otherwise the minimum radicand, ties to the smallest node index.  The reference keeps the first node it
meets at the minimum distance, so its index is only pinned to the tie set: the nodes at exactly that distance.

The point sets are the inputs where grid-indexed kernels go wrong: a pile of identical points and scattered pairs,
an integer lattice with radii on lattice distances, flat and collinear sets, far outliers and non-finite nodes.
Insertion order is shuffled with a fixed seed, so that the reference's kd tree (and its recursion) stays shallow.
"""
from __future__ import annotations

import math

import numpy as np

BOX = 20.0
N_POINTS = 20000
PILE = 300                      # > 256: cell_sort_kernel leaves the cell unsorted, the v5 octet table overflows


def radicands(pts, q):
    """Radicand of euclidianDist from the query q to every row of pts, reference operation order."""
    s = np.zeros(len(pts))
    with np.errstate(over="ignore", invalid="ignore"):
        for k in range(pts.shape[1]):
            dk = q[k] - pts[:, k]
            s = s + dk * dk
    return s


def nearest(pts, q):
    """(node, dist, tie set) by the device's rule; the tie set holds every node at exactly that distance."""
    s = radicands(pts, np.asarray(q, dtype=np.float64))
    if np.isnan(s[0]):
        return 0, float(np.sqrt(s[0])), np.array([0])
    smin = np.min(np.where(np.isnan(s), np.inf, s))
    i = int(np.flatnonzero(s == smin)[0])
    d = float(np.sqrt(smin))
    return i, d, np.flatnonzero(np.sqrt(s) == d)


def range_query(pts, q, r):
    """kdFindWithinRange(tree, r, q) -> (node indices ascending, keys)."""
    dist = np.sqrt(radicands(pts, np.asarray(q, dtype=np.float64)))
    hit = dist < r
    hit[0] = dist[0] <= r
    idx = np.flatnonzero(hit)
    return idx, dist[idx]


# ------------------------------------------------------------------------------------------------ point sets
def _uniform(rng, n, d, box=BOX):
    return rng.uniform(-box, box, (n, d))


def _shuffled(rng, pts, first=None):
    """Shuffle the insertion order; `first` (a row) becomes the root."""
    pts = pts[rng.permutation(len(pts))]
    if first is not None:
        pts = np.vstack([np.asarray(first, dtype=np.float64)[None, :], pts])
    return np.ascontiguousarray(pts)


def grid_dims(pts, occupancy=4.0, aspect=2.0):
    """Cells per axis of the device's grid index over pts (tree_reindex in csrc/tree.cu): axes whose bbox is flat or
    not finite get one cell.  Returns (lo, cell, dims) of the first three axes."""
    d = pts.shape[1]
    mn, mx = np.zeros(3), np.zeros(3)
    for k in range(3):
        col = pts[:, k] if k < d else np.zeros(1)
        col = col[~np.isnan(col)]
        mn[k], mx[k] = (col.min(), col.max()) if len(col) else (0.0, 0.0)
        if not (np.isfinite(mn[k]) and np.isfinite(mx[k])):
            mn[k] = mx[k] = 0.0
    with np.errstate(over="ignore"):
        ext = mx - mn
    ext = np.where((np.arange(3) < d) & (ext > 0) & np.isfinite(ext), ext, 0.0)
    nonflat = int(np.count_nonzero(ext > 0))
    dims = [1, 1, 1]
    if nonflat:
        vol = float(np.prod(ext[ext > 0]))
        c = math.pow(vol / max(1.0, len(pts) / max(0.25, occupancy)), 1.0 / nonflat)
        cs = [c, c, c]
        if ext[0] > 0 and nonflat >= 2 and aspect > 1.0:
            cs[0] = c / math.pow(aspect, (nonflat - 1.0) / nonflat)
            cs[1] = cs[2] = c * math.pow(aspect, 1.0 / nonflat)
        dims = [min(1024, max(1, math.ceil(ext[k] / cs[k]))) if ext[k] > 0 else 1 for k in range(3)]
    cell = np.where(ext > 0, ext / np.array(dims), 1.0)
    return mn, cell, dims


def cross_boundary_case(pts, q_x=10.0):
    """Deterministic case for a nearest search that trusts the extent of a boundary cell: a query at x = q_x just
    below a y-cell boundary, one point inside its own cell 0.3 away and one just across the boundary 0.01 away.
    Nodes within 1 of the query are moved away first.  Returns (points, query, index of the nearest)."""
    lo, cell, dims = grid_dims(np.vstack([pts, pts[1:3]]))     # the two points added below keep the bbox
    zc = lo[2] + (dims[2] // 2 + 0.5) * cell[2]
    b = lo[1] + (dims[1] // 2) * cell[1]                  # a y-cell boundary near the middle
    q = np.array([q_x, b - 0.005, zc] + [0.0] * (pts.shape[1] - 3))
    far = np.sqrt(radicands(pts, q)) < 1.0
    far[0] = False
    pts = pts.copy()
    pts[far, 0] -= 5.0
    a = q.copy(); a[1] -= 0.3
    c = q.copy(); c[1] += 0.01
    pts = np.vstack([pts, a[None, :], c[None, :]])
    return np.ascontiguousarray(pts), q, len(pts) - 1


def point_set(name, seed=7):
    """(points, queries, radius, case) of one degenerate set.  Queries: uniform over a box slightly larger than the
    points' and, in front, every node among the first 200, the special placements of the set and a NaN, an inf and a
    1e200 query.  case: (query, expected nearest node) of cross_boundary_case, or None."""
    rng = np.random.default_rng(seed)
    d = 3
    specials = []
    r = 1.1
    if name == "duplicates":
        base = _uniform(rng, N_POINTS - PILE - 1000, d)
        pile = np.tile(np.array([1.25, -3.5, 2.0]), (PILE, 1))
        pairs = _uniform(rng, 500, d)
        pts = _shuffled(rng, np.vstack([base, pile, pairs, pairs]))
        specials = [pile[0], pile[0] + 1e-9, pile[0] + [0.3, 0.0, 0.0], pairs[0], pairs[1]]
    elif name.startswith("lattice"):
        d = int(name[-1])
        side = {2: 120, 3: 24, 4: 11}[d]
        axes = np.meshgrid(*[np.arange(side, dtype=np.float64) - side // 2] * d, indexing="ij")
        pts = _shuffled(rng, np.stack([a.ravel() for a in axes], axis=1))
        r = 5.0
        root = pts[0]
        off = np.zeros(d)
        for o in ([3.0, 4.0], [4.0, 3.0], [5.0, 0.0], [1.0, 0.0], [1.0, 1.0], [0.5, 0.5]):
            off[:2] = o
            specials += [root + off, root - off]
        specials += list(pts[1:101] + 0.5) + list(pts[101:151] + np.r_[0.5, np.zeros(d - 1)])   # 2^d- and 2-way ties
    elif name == "flat":
        pts = _uniform(rng, N_POINTS, d)
        pts[:, 2] = 1.5
        pts = _shuffled(rng, pts)
        specials = [[0.0, 0.0, 1.5], [3.0, -2.0, 1.5 + 1e-12], [3.0, -2.0, 0.5]]
    elif name == "collinear":
        t = rng.uniform(-BOX, BOX, N_POINTS)
        pts = _shuffled(rng, np.stack([t, 2.0 * t, -t], axis=1))
        specials = [[1.0, 2.0, -1.0], [1.0, 2.5, -1.0], [0.0, 0.0, 0.0]]
    elif name == "collinear_axis":
        t = rng.uniform(-BOX, BOX, N_POINTS)
        pts = _shuffled(rng, np.stack([t, np.full_like(t, -2.0), np.full_like(t, 3.0)], axis=1))
        specials = [[1.0, -2.0, 3.0], [1.0, -1.5, 3.0], [30.0, -2.0, 3.0]]
    elif name in ("outlier_1e6", "outlier_1e30"):
        far = 1e6 if name == "outlier_1e6" else 1e30
        pts = _shuffled(rng, np.vstack([_uniform(rng, N_POINTS - 1, d), [[far, -far, far]]]))
        specials = [[far, -far, far], [far * 0.999, -far, far]]
    elif name in ("nan_node", "posinf_node", "neginf_node"):
        v = {"nan_node": np.nan, "posinf_node": np.inf, "neginf_node": -np.inf}[name]
        extra = [[v, 0.5, 0.5], [1.0, 2.0, v]] if name == "nan_node" else [[v, 0.5, 0.5]]   # +-inf: x flat only
        pts = _shuffled(rng, np.vstack([_uniform(rng, N_POINTS - len(extra), d), extra]))
        specials = extra + [[v, v, v], [1.0, v, 2.0]]
    elif name == "overflow_extent":
        pts = _shuffled(rng, np.vstack([_uniform(rng, N_POINTS - 2, d), [[1e308, 0.0, 0.0], [-1e308, 1.0, 1.0]]]))
        specials = [[1e308, 0.0, 0.0], [-1e308, 1.0, 1.0], [0.0, 1e308, 0.0]]
    elif name == "nan_root":
        pts = _shuffled(rng, _uniform(rng, N_POINTS - 1, d), first=[np.nan, 1.0, 2.0])
    else:
        raise KeyError(name)
    case = None
    if name in ("posinf_node", "neginf_node", "overflow_extent"):   # x has one cell: the cell-boundary case
        pts, cq, ci = cross_boundary_case(pts)
        specials.append(cq)
        case = (cq, ci)
    qbox = (side // 2 + 1.0) if name.startswith("lattice") else BOX * 1.05
    qs = _uniform(np.random.default_rng(seed + 1), 4400, d, qbox)
    front = [pts[i] for i in range(min(200, len(pts)))] + [np.asarray(s, dtype=np.float64) for s in specials]
    front += [np.full(d, np.nan), np.r_[np.inf, np.zeros(d - 1)], np.full(d, 1e200)]
    qs[:len(front)] = np.array(front)
    return np.ascontiguousarray(pts), np.ascontiguousarray(qs), r, case


SETS = ["duplicates", "lattice2", "lattice3", "lattice4", "flat", "collinear", "collinear_axis", "outlier_1e6",
        "outlier_1e30", "nan_node", "posinf_node", "neginf_node", "overflow_extent", "nan_root"]


def radii_for(name, r):
    """Uniform radii of a set: the lattice gets the lattice distances 1, sqrt(2) and 5 exactly (hits need <)."""
    if name.startswith("lattice"):
        return [1.0, math.sqrt(2.0), 5.0]
    return [r]
