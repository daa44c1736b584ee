"""Brute-force model of kdFindWithinRange / kdFindNearest on trees with wrap-around dimensions, plain numpy float64.

It restates the reference's rule without any tree: the ghost identities of a query in the order of getNextGhostPoint
(ghostPoint.jl:60-111), each used only when the point of the unwrapped space closest to it is within the current
bound (:104); the range list is the union over the identities with the key of the FIRST identity that reaches a node
(addToRangeList dedup, kdTree_general.jl:765-771, 903-916); the root is admitted with <= by the real identity only
(:895-898); nearest keeps the real identity's minimum and lets a ghost replace it only when strictly closer
(:357-385).  Distances are euclidianDist: a left-to-right sum of squares and one sqrt, no FMA.

The wrap configurations and the edge placements shared by test_wrap_model.py (model vs CPU oracle) and
test_gpu_wrap.py (model and oracle vs the device) live here too.
"""
from __future__ import annotations

import numpy as np

TWO_PI = 2.0 * np.pi

# (d, wraps (0-based dims), periods, box of the non-wrapped dims {dim: (lo, hi)})
CONFIGS = {
    "c4_theta": (4, [3], [TWO_PI], {0: (-10.0, 10.0), 1: (-10.0, 10.0), 2: (0.0, 0.0)}),
    "testGhost_z": (3, [2], [TWO_PI], {0: (-8.0, 8.0), 1: (-8.0, 8.0)}),
    "torus_xy": (2, [0, 1], [1.0, 1.0], {}),
    "x_and_z": (3, [0, 2], [4.0, TWO_PI], {1: (-5.0, 5.0)}),
    "three_wraps": (4, [0, 1, 3], [3.0, 3.0, TWO_PI], {2: (-3.0, 3.0)}),
    "max_wraps": (4, [0, 1, 2, 3], [2.0, 2.0, 2.0, TWO_PI], {}),
}

RADIUS_FACTORS = (0.1, 0.37, 0.5, "next_half", 0.55, 0.8, 1.3)


def radii(periods):
    """The radii of the wrap tests for a tree whose shortest period is min(periods): both sides of the P/2 bound
    of the ghost-pair path, and 1.3 P, where several identities reach the same node."""
    pmin = float(min(periods))
    out = []
    for f in RADIUS_FACTORS:
        out.append(float(np.nextafter(pmin / 2.0, np.inf)) if f == "next_half" else f * pmin)
    return out


def euclid(a, P):
    """euclidianDist of one point a to every row of P: left-to-right sum of squares, one sqrt."""
    s = np.zeros(len(P))
    for k in range(P.shape[1]):
        dk = a[k] - P[:, k]
        s = s + dk * dk
    return np.sqrt(s)


def _radicand(a, P):
    s = np.zeros(len(P))
    for k in range(P.shape[1]):
        dk = a[k] - P[:, k]
        s = s + dk * dk
    return s


def ghosts(q, wraps, wps, bound):
    """The used ghost identities of q in the reference's order; bound() is re-read before each ghost."""
    w = len(wraps)
    for p in range(1, 1 << w):          # bit b of p shifts wraps[w-1-b]
        g, c = q.copy(), q.copy()
        for b in range(w):
            if (p >> b) & 1:
                wi = w - 1 - b
                dim, P = wraps[wi], wps[wi]
                if q[dim] < P / 2.0:
                    g[dim], c[dim] = q[dim] + P, P
                else:
                    g[dim], c[dim] = q[dim] - P, 0.0
        if euclid(c, g[None, :])[0] > bound():
            continue
        yield g


def range_query(pts, q, r, wraps, wps):
    """kdFindWithinRange(tree, r, q) -> (node indices ascending, keys)."""
    q = np.asarray(q, dtype=np.float64)
    n = len(pts)
    key = np.zeros(n)
    taken = np.zeros(n, dtype=bool)
    d0 = euclid(q, pts[:1])[0]
    if d0 <= r:
        taken[0], key[0] = True, d0
    for ident in [q] + list(ghosts(q, wraps, wps, lambda: r)):
        dist = euclid(ident, pts)
        m = (dist < r) & ~taken
        key[m] = dist[m]
        taken |= m
    idx = np.nonzero(taken)[0]
    return idx, key[idx]


def nearest(pts, q, wraps, wps):
    """kdFindNearest(tree, q) -> (node, dist).  Within one identity the smallest radicand wins and ties go to the
    smallest node index (the device's documented tie rule); across identities a later one must be strictly closer."""
    q = np.asarray(q, dtype=np.float64)
    best = [0, euclid(q, pts[:1])[0]]   # the reference starts from the root

    def consider(ident):
        s = _radicand(ident, pts)
        if not np.any(s == s):
            return
        smin = np.nanmin(s)
        d = np.sqrt(smin)
        if d < best[1]:
            best[0], best[1] = int(np.nonzero(s == smin)[0][0]), d

    consider(q)
    for g in ghosts(q, wraps, wps, lambda: best[1]):
        consider(g)
    return best[0], best[1]


# ------------------------------------------------------------------------------------------------- placements
def wrap_specials(P):
    """Wrap coordinates where the ghost rule changes: exactly 0, P/2 and P, just below P/2, within 1e-12 of the
    seam on both sides, and slightly outside [0, P) (the reference does not normalise; Dubins saturate clamps into
    [0, 2 pi] inclusive)."""
    half = P / 2.0
    return np.array([0.0, half, np.nextafter(half, 0.0), P, 1e-12, P - 1e-12, -1e-12, P + 1e-12,
                     np.nextafter(0.0, -1.0), np.nextafter(P, np.inf), -1e-3 * P, P * (1.0 + 1e-3)])


def uniform(seed, n, cfg):
    d, wraps, wps, box = cfg
    rng = np.random.default_rng(seed)
    u = rng.random((n, d))
    out = np.zeros((n, d))
    for k in range(d):
        if k in wraps:
            lo, hi = 0.0, wps[wraps.index(k)]
        else:
            lo, hi = box[k]
        out[:, k] = lo + (hi - lo) * u[:, k]
    return out


def with_edges(a, cfg, first=0):
    """Overwrite rows first.. of a with every special wrap coordinate on every wrap dimension, alone and mixed."""
    d, wraps, wps, _ = cfg
    sp = [wrap_specials(P) for P in wps]
    m = len(sp[0])
    row = first
    for wi in range(len(wraps)):            # one wrap dimension special, the others uniform
        for v in sp[wi]:
            a[row, wraps[wi]] = v
            row += 1
    for k in range(m):                      # every wrap dimension special at once, mixed
        for wi in range(len(wraps)):
            a[row, wraps[wi]] = sp[wi][(k + 5 * wi) % m]
        row += 1
    return row


def points(seed, n, cfg):
    p = uniform(seed, n, cfg)
    with_edges(p, cfg, first=1)             # keep a uniform root
    return np.ascontiguousarray(p)


def queries(seed, n, cfg, pts):
    """Uniform queries with the edge placements in front, a query exactly on the root and one NaN query."""
    q = uniform(seed, n, cfg)
    row = with_edges(q, cfg) if n > 64 else 0
    if n >= 3:
        q[min(row, n - 2)] = pts[0]
        q[min(row + 1, n - 1)] = np.nan
    return np.ascontiguousarray(q)


def tie_tree(cfg):
    """Tree [far root, B, A] plus far points, the query, and A's index."""
    d, wraps, wps, _ = cfg
    w0, P = wraps[0], wps[0]
    base = uniform(9, 1, cfg)[0]
    base[w0] = 0.0
    other = [k for k in range(d) if k != w0][0]
    q = base.copy()
    q[other] += 0.01 * min(wps)
    A = base.copy()
    B = base.copy()
    B[w0] = P
    far = uniform(10, 200, cfg)
    keep = euclid(q, far) > 0.2 * min(wps)
    for g in ghosts(q, wraps, wps, lambda: np.inf):
        keep &= euclid(g, far) > 0.2 * min(wps)
    root = far[keep][:1]
    pts = np.ascontiguousarray(np.vstack([root, B[None], A[None], far[keep][1:40]]))
    return pts, q, 2
