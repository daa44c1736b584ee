"""Handle objects over the C ABI (one class per opaque handle of rrtqx_b200.h).

These are the batched, index-based calls.  The reference-shaped API
(KDTree / kdInsert / kdFindWithinRange / explicitEdgeCheck / addNewObstacle ...)
is layered on top in kdtree.py, collision.py and sweep.py.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _abi as A


class Context:
    """rrtqx_ctx: one CUDA device + stream.  Raises if no B200 is usable."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self.L = A.lib()
        h = A.vp()
        A.check(self.L.rrtqx_ctx_create(int(device), stream, C.byref(h)), None)
        self.h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "h", None):
            self.L.rrtqx_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        A.check(self.L.rrtqx_ctx_sync(self.h), self.h)

    def host_array(self, shape, dtype):
        """A numpy array over page-locked host memory from rrtqx_host_alloc (freed when the array's owner dies)."""
        shape = (int(shape),) if np.isscalar(shape) else tuple(int(x) for x in shape)
        dtype = np.dtype(dtype)
        nbytes = int(np.prod(shape)) * dtype.itemsize
        p = A.vp()
        A.check(self.L.rrtqx_host_alloc(self.h, max(nbytes, 1), C.byref(p)), self.h)
        buf = (C.c_char * max(nbytes, 1)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
        L, addr = self.L, p.value
        import weakref
        weakref.finalize(buf, lambda: L.rrtqx_host_free(None, addr))
        return arr

    def reload_tuning(self):
        """Re-read the diagnostic RRTQX_* environment switches (they are otherwise read once, at creation)."""
        A.check(self.L.rrtqx_ctx_reload_tuning(self.h), self.h)

    def kernel_launches(self) -> int:
        n = A.i64(0)
        A.check(self.L.rrtqx_ctx_kernel_launches(self.h, C.byref(n)), self.h)
        return int(n.value)

    def measure_fp64_peak(self) -> float:
        """Measured FP64 FMA throughput in TFLOP/s (roofline denominator of the FP64-bound collision kernels)."""
        v = A.f64(0.0)
        A.check(self.L.rrtqx_ctx_measure_fp64_peak(self.h, C.byref(v)), self.h)
        return float(v.value)

    def last_phase_ms(self, phase: str) -> float:
        ms = C.c_float(0.0)
        A.check(self.L.rrtqx_ctx_last_phase_ms(self.h, phase.encode(), C.byref(ms)), self.h)
        return float(ms.value)


class RangeResult:
    """rrtqx_range_result: device-resident neighbour lists of a query batch."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self.L = ctx.L
        self.h = A.vp()  # NULL until the first query fills it

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.L.rrtqx_range_result_destroy(self.h)
            self.h = A.vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sizes(self):
        nq, tot = A.i64(0), A.i64(0)
        A.check(self.L.rrtqx_range_result_sizes(self.h, C.byref(nq), C.byref(tot)), self.ctx.h)
        return int(nq.value), int(tot.value)

    def layout(self):
        nq, _ = self.sizes()
        counts = np.empty(nq, dtype=np.int32)
        offsets = np.empty(nq, dtype=np.int64)
        A.check(self.L.rrtqx_range_result_layout(self.h, A.ptr(counts), A.ptr(offsets)), self.ctx.h)
        return counts, offsets

    def fetch(self, want_dist=True, idx_out=None, dist_out=None):
        _, tot = self.sizes()
        idx = np.empty(tot, dtype=np.int32) if idx_out is None else idx_out
        dist = (np.empty(tot, dtype=np.float64) if dist_out is None else dist_out) if want_dist else None
        A.check(self.L.rrtqx_range_result_fetch(self.h, A.ptr(idx), A.ptr(dist)), self.ctx.h)
        return idx, dist

    def device_pointers(self):
        p = [A.vp() for _ in range(4)]
        A.check(self.L.rrtqx_range_result_device(self.h, *[C.byref(x) for x in p]), self.ctx.h)
        return tuple(x.value for x in p)  # counts, offsets, idx, dist

    def lists(self, want_dist=True):
        """Python-side view: list of (idx array, dist array) per query."""
        counts, offsets = self.layout()
        idx, dist = self.fetch(want_dist)
        out = []
        for c, o in zip(counts, offsets):
            out.append((idx[o:o + c], dist[o:o + c] if dist is not None else None))
        return out


class DeviceTree:
    """rrtqx_tree: the GPU-resident KDTree (points + kd topology + grid index)."""

    def __init__(self, ctx: Context, d: int, wraps=(), wrap_points=()):
        self.ctx = ctx
        self.L = ctx.L
        self.d = int(d)
        w = np.asarray(list(wraps), dtype=np.int32)
        wp = np.asarray(list(wrap_points), dtype=np.float64)
        assert w.size == wp.size
        h = A.vp()
        A.check(self.L.rrtqx_tree_create(ctx.h, self.d, int(w.size), A.ptr(w) if w.size else None,
                                         A.ptr(wp) if wp.size else None, C.byref(h)), ctx.h)
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.rrtqx_tree_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        n = A.i64(0)
        A.check(self.L.rrtqx_tree_size(self.h, C.byref(n)), self.ctx.h)
        return int(n.value)

    def insert_batch(self, positions, n=None) -> int:
        """kdInsert for every row, in order; returns the index of the first."""
        if isinstance(positions, np.ndarray) or not hasattr(positions, "data_ptr"):
            positions = A.as_f64(positions, self.d)
            n = positions.shape[0]
        first = A.i32(0)
        A.check(self.L.rrtqx_tree_insert_batch(self.h, A.ptr(positions), int(n), C.byref(first)), self.ctx.h)
        return int(first.value)

    def insert(self, position) -> int:
        p = A.as_f64(position).reshape(-1)
        assert p.size == self.d
        idx = A.i32(0)
        A.check(self.L.rrtqx_tree_insert(self.h, A.ptr(p), C.byref(idx)), self.ctx.h)
        return int(idx.value)

    def kd_fields(self, first=0, count=None):
        if count is None:
            count = len(self) - first
        out = [np.empty(count, dtype=np.int32) for _ in range(4)]
        A.check(self.L.rrtqx_tree_kd_fields(self.h, first, count, *[A.ptr(a) for a in out]), self.ctx.h)
        return tuple(out)  # parent, childL, childR, split

    def positions(self, first=0, count=None):
        if count is None:
            count = len(self) - first
        out = np.empty((count, self.d), dtype=np.float64)
        A.check(self.L.rrtqx_tree_positions(self.h, first, count, A.ptr(out)), self.ctx.h)
        return out

    def preorder(self):
        """Node indices in the visit order of the reference's recursive kd traversals (dump row order)."""
        out = np.empty(len(self), dtype=np.int32)
        A.check(self.L.rrtqx_tree_preorder(self.h, A.ptr(out)), self.ctx.h)
        return out

    def set_cell_occupancy(self, ppc: float):
        A.check(self.L.rrtqx_tree_set_cell_occupancy(self.h, float(ppc)), self.ctx.h)

    def reindex(self):
        A.check(self.L.rrtqx_tree_reindex(self.h), self.ctx.h)

    def range_query(self, queries, r, ranges=None, want_dist=True, count_only=False, result: RangeResult | None = None,
                    n_queries=None):
        """Batched kdFindWithinRange.  queries: (nq x d) numpy array or a device
        pointer/tensor (then pass n_queries).  Returns (RangeResult, total)."""
        if isinstance(queries, np.ndarray) or not (hasattr(queries, "data_ptr") or isinstance(queries, int)):
            queries = A.as_f64(queries, self.d)
            n_queries = queries.shape[0]
        if ranges is not None and isinstance(ranges, (list, tuple, np.ndarray)):
            ranges = A.as_f64(ranges).reshape(-1)
            assert ranges.size == n_queries
        if result is None:
            result = RangeResult(self.ctx)
        flags = (A.RANGE_WANT_DIST if want_dist else 0) | (A.RANGE_COUNT_ONLY if count_only else 0)
        total = A.i64(0)
        A.check(self.L.rrtqx_range_query_batch(self.h, A.ptr(queries), int(n_queries), float(r), A.ptr(ranges), flags,
                                               C.byref(result.h), C.byref(total)), self.ctx.h)
        return result, int(total.value)

    def nearest(self, queries, n_queries=None, idx_out=None, dist_out=None):
        """Batched kdFindNearest -> (idx int32[nq], dist float64[nq])."""
        if isinstance(queries, np.ndarray) or not (hasattr(queries, "data_ptr") or isinstance(queries, int)):
            queries = A.as_f64(queries, self.d)
            n_queries = queries.shape[0]
        idx = np.empty(n_queries, dtype=np.int32) if idx_out is None else idx_out
        dist = np.empty(n_queries, dtype=np.float64) if dist_out is None else dist_out
        A.check(self.L.rrtqx_nearest_batch(self.h, A.ptr(queries), int(n_queries), A.ptr(idx), A.ptr(dist)), self.ctx.h)
        return idx, dist


class SphereSet:
    """rrtqx_spheres: CSpace.obstacles (List{SphereObstacle}) flattened."""

    def __init__(self, ctx: Context, centers=None, radii=None, active=None):
        self.ctx = ctx
        self.L = ctx.L
        h = A.vp()
        A.check(self.L.rrtqx_spheres_create(ctx.h, C.byref(h)), ctx.h)
        self.h = h
        if centers is not None:
            self.upload(centers, radii, active)

    def close(self):
        if getattr(self, "h", None):
            self.L.rrtqx_spheres_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        n = A.i64(0)
        A.check(self.L.rrtqx_spheres_size(self.h, C.byref(n)), self.ctx.h)
        return int(n.value)

    def upload(self, centers, radii, active=None):
        centers = A.as_f64(centers, 3)
        n = centers.shape[0]
        radii = np.ascontiguousarray(np.broadcast_to(np.asarray(radii, dtype=np.float64), (n,)))
        act = None if active is None else A.as_u8(np.asarray(active).astype(np.uint8))
        A.check(self.L.rrtqx_spheres_upload(self.h, A.ptr(centers) if n else None, A.ptr(radii) if n else None,
                                            A.ptr(act), n), self.ctx.h)

    def update(self, first, radii=None, active=None):
        count = len(radii) if radii is not None else len(active)
        r = None if radii is None else A.as_f64(radii).reshape(-1)
        a = None if active is None else A.as_u8(np.asarray(active).astype(np.uint8))
        A.check(self.L.rrtqx_spheres_update(self.h, int(first), int(count), A.ptr(r), A.ptr(a)), self.ctx.h)


def edge_check_batch(tree: DeviceTree, spheres: SphereSet, src, dst, robot_radius, flags=0, n_edges=None, out=None):
    """Batched explicitEdgeCheck(S, edge) over edges between tree nodes."""
    if isinstance(src, np.ndarray) or isinstance(src, (list, tuple)):
        src, dst = A.as_i32(src), A.as_i32(dst)
        n_edges = src.size
    if out is None:
        out = np.empty(n_edges, dtype=np.uint8)
    A.check(tree.L.rrtqx_edge_check_batch(tree.h, spheres.h, A.ptr(src), A.ptr(dst), int(n_edges), float(robot_radius),
                                          int(flags), A.ptr(out)), tree.ctx.h)
    return out


def segment_check_batch(ctx: Context, spheres: SphereSet, starts, ends, robot_radius, flags=0):
    starts, ends = A.as_f64(starts, 3), A.as_f64(ends, 3)
    n = starts.shape[0]
    out = np.empty(n, dtype=np.uint8)
    A.check(ctx.L.rrtqx_segment_check_batch(ctx.h, spheres.h, A.ptr(starts), A.ptr(ends), n, float(robot_radius),
                                            int(flags), A.ptr(out)), ctx.h)
    return out


def node_check_batch(ctx: Context, spheres: SphereSet, points, robot_radius, flags=0):
    """Batched explicitPointCheck -> (collide uint8[n], certificate float64[n])."""
    points = A.as_f64(points, 3)
    n = points.shape[0]
    out = np.empty(n, dtype=np.uint8)
    cert = np.empty(n, dtype=np.float64)
    A.check(ctx.L.rrtqx_node_check_batch(ctx.h, spheres.h, A.ptr(points), n, float(robot_radius), int(flags),
                                         A.ptr(out), A.ptr(cert)), ctx.h)
    return out, cert


class SweepResult:
    def __init__(self, ctx: Context):
        self.ctx = ctx
        self.L = ctx.L
        self.h = A.vp()

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.L.rrtqx_sweep_result_destroy(self.h)
            self.h = A.vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sizes(self):
        v = [A.i64(0) for _ in range(4)]
        A.check(self.L.rrtqx_sweep_result_sizes(self.h, *[C.byref(x) for x in v]), self.ctx.h)
        return tuple(int(x.value) for x in v)  # edge_hits, node_hits, candidates, pair_tests

    def fetch(self):
        ne, nn, _, _ = self.sizes()
        e = np.empty(ne, dtype=np.int32)
        n = np.empty(nn, dtype=np.int32)
        A.check(self.L.rrtqx_sweep_result_fetch(self.h, A.ptr(e), A.ptr(n)), self.ctx.h)
        return e, n

    def flags(self, n_edges: int, n_nodes: int):
        """The same result as byte flags: edge_flag[n_edges], node_flag[n_nodes] (sizes of the swept edge set)."""
        ef = np.empty(int(n_edges), dtype=np.uint8)
        nf = np.empty(int(n_nodes), dtype=np.uint8)
        A.check(self.L.rrtqx_sweep_result_flags(self.h, A.ptr(ef), A.ptr(nf)), self.ctx.h)
        return ef, nf


class EdgeSet:
    """rrtqx_edges: device mirror of the planner's out-edge lists + parents."""

    def __init__(self, tree: DeviceTree):
        self.tree = tree
        self.ctx = tree.ctx
        self.L = tree.L
        h = A.vp()
        A.check(self.L.rrtqx_edges_create(tree.h, C.byref(h)), self.ctx.h)
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.rrtqx_edges_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        n = A.i64(0)
        A.check(self.L.rrtqx_edges_size(self.h, C.byref(n)), self.ctx.h)
        return int(n.value)

    def upload(self, src, dst, parent=None, n_edges=None):
        if isinstance(src, (np.ndarray, list, tuple)):
            src, dst = A.as_i32(src), A.as_i32(dst)
            n_edges = src.size
        par = None if parent is None else A.as_i32(parent)
        A.check(self.L.rrtqx_edges_upload(self.h, A.ptr(src), A.ptr(dst), int(n_edges), A.ptr(par),
                                          0 if par is None else par.size), self.ctx.h)

    def append(self, src, dst):
        """Edges created since the upload (ids continue the upload order); no re-upload of the graph."""
        src, dst = A.as_i32(src), A.as_i32(dst)
        A.check(self.L.rrtqx_edges_append(self.h, A.ptr(src), A.ptr(dst), len(src)), self.ctx.h)

    def set_parents(self, node_ids, parent_ids):
        """makeParentOf for a batch of nodes: parent_ids[i] (or -1) becomes the parent of node_ids[i]."""
        node_ids, parent_ids = A.as_i32(node_ids), A.as_i32(parent_ids)
        A.check(self.L.rrtqx_edges_set_parents(self.h, A.ptr(node_ids), A.ptr(parent_ids), len(node_ids)), self.ctx.h)

    def check_all(self, spheres: SphereSet, robot_radius, flags=0, out=None):
        """explicitEdgeCheck(S, edge) of every resident out-edge -> uint8[n_edges] (edge id order)."""
        if out is None:
            out = np.empty(len(self), dtype=np.uint8)
        A.check(self.L.rrtqx_edges_check_batch(self.h, spheres.h, float(robot_radius), int(flags), A.ptr(out)), self.ctx.h)
        return out

    def add_sweep(self, spheres: SphereSet, ob_ids, robot_radius, delta, flags=0, result: SweepResult | None = None):
        ob_ids = A.as_i32(ob_ids)
        if result is None:
            result = SweepResult(self.ctx)
        A.check(self.L.rrtqx_obstacle_add_sweep(self.h, spheres.h, A.ptr(ob_ids), ob_ids.size, float(robot_radius),
                                                float(delta), int(flags), C.byref(result.h)), self.ctx.h)
        return result

    def remove_sweep(self, spheres: SphereSet, ob_id, other_ids, edge_dist_inf, robot_radius, delta, flags=0,
                     result: SweepResult | None = None):
        other_ids = A.as_i32(other_ids)
        inf = A.as_u8(np.asarray(edge_dist_inf).astype(np.uint8))
        if result is None:
            result = SweepResult(self.ctx)
        A.check(self.L.rrtqx_obstacle_remove_sweep(self.h, spheres.h, int(ob_id), A.ptr(other_ids) if other_ids.size else None,
                                                   other_ids.size, A.ptr(inf), float(robot_radius), float(delta),
                                                   int(flags), C.byref(result.h)), self.ctx.h)
        return result


    # ---- DubinsEdge world (Otte generation, DRRT.jl:3048-3268) -------------------------------------------
    def set_trajectories(self, traj_ptr, traj_xy):
        """Upload edge.trajectory[:,1:2] of every ITEM (out-edges in upload order, then one parent edge per node)
        as a CSR: traj_ptr[n_edges + n_nodes + 1], traj_xy rows x 2."""
        if isinstance(traj_ptr, (np.ndarray, list, tuple)):
            traj_ptr = np.ascontiguousarray(traj_ptr, dtype=np.int64)
            traj_xy = A.as_f64(traj_xy, 2)
        A.check(self.L.rrtqx_edges_set_trajectories(self.h, A.ptr(traj_ptr), A.ptr(traj_xy) if traj_xy is not None and
                                                    (not isinstance(traj_xy, np.ndarray) or traj_xy.size) else None), self.ctx.h)

    def solve_trajectories(self, min_turn_radius) -> int:
        """calculateTrajectory of every item on the device (DRRT_DubinsEdge_functions.jl:329-709); returns the rows."""
        n = A.i64(0)
        A.check(self.L.rrtqx_edges_solve_trajectories(self.h, float(min_turn_radius), C.byref(n)), self.ctx.h)
        return int(n.value)

    def trajectories(self):
        """Resident trajectories copied to the host: (traj_ptr int64[items + 1], traj_xy float64[rows, 2])."""
        ni, nr = A.i64(0), A.i64(0)
        A.check(self.L.rrtqx_edges_trajectories_device(self.h, None, None, C.byref(ni), C.byref(nr)), self.ctx.h)
        ptr = np.empty(ni.value + 1, dtype=np.int64)
        xy = np.empty((nr.value, 2), dtype=np.float64)
        A.check(self.L.rrtqx_edges_trajectories_fetch(self.h, A.ptr(ptr), A.ptr(xy) if xy.size else None), self.ctx.h)
        return ptr, xy

    def add_sweep_2d(self, polys, ob_ids, robot_radius, delta, min_turn_radius, flags=0, result: SweepResult | None = None):
        ob_ids = A.as_i32(ob_ids)
        if result is None:
            result = SweepResult(self.ctx)
        A.check(self.L.rrtqx_obstacle_add_sweep_2d(self.h, polys.h, A.ptr(ob_ids), ob_ids.size, float(robot_radius),
                                                   float(delta), float(min_turn_radius), int(flags), C.byref(result.h)),
                self.ctx.h)
        return result

    def remove_sweep_2d(self, polys, ob_id, other_ids, edge_dist_inf, robot_radius, delta, min_turn_radius, flags=0,
                        result: SweepResult | None = None):
        other_ids = A.as_i32(other_ids)
        inf = A.as_u8(np.asarray(edge_dist_inf).astype(np.uint8))
        if result is None:
            result = SweepResult(self.ctx)
        A.check(self.L.rrtqx_obstacle_remove_sweep_2d(self.h, polys.h, int(ob_id), A.ptr(other_ids) if other_ids.size else None,
                                                      other_ids.size, A.ptr(inf), float(robot_radius), float(delta),
                                                      float(min_turn_radius), int(flags), C.byref(result.h)), self.ctx.h)
        return result


class ExtendResult:
    """Outputs of one rrtqx_extend_query call."""
    __slots__ = ("nearest_idx", "nearest_dist", "point_collides", "point_cert", "count", "idx", "dist", "fwd", "rev")


def extend_query(tree: DeviceTree, spheres: SphereSet, point, r, robot_radius, flags=0, capacity=4096, bufs=None):
    """One planner iteration's geometric work in one launch (rrtqx.jl:926-950, DRRT_Q.jl:2546-2641)."""
    p = A.as_f64(point).reshape(-1)
    if bufs is None or len(bufs[0]) < capacity:
        bufs = (np.empty(capacity, dtype=np.int32), np.empty(capacity, dtype=np.float64),
                np.empty(capacity, dtype=np.uint8), np.empty(capacity, dtype=np.uint8))
    ni, nd, pc, ce, cnt = A.i32(0), A.f64(0.0), C.c_uint8(0), A.f64(0.0), A.i32(0)
    A.check(tree.L.rrtqx_extend_query(tree.h, spheres.h, A.ptr(p), float(r), float(robot_radius), int(flags), int(capacity),
                                      C.byref(ni), C.byref(nd), C.byref(pc), C.byref(ce), C.byref(cnt), A.ptr(bufs[0]),
                                      A.ptr(bufs[1]), A.ptr(bufs[2]), A.ptr(bufs[3])), tree.ctx.h)
    out = ExtendResult()
    out.nearest_idx, out.nearest_dist = int(ni.value), float(nd.value)
    out.point_collides, out.point_cert, out.count = bool(pc.value), float(ce.value), int(cnt.value)
    m = min(out.count, capacity)
    out.idx, out.dist, out.fwd, out.rev = bufs[0][:m], bufs[1][:m], bufs[2][:m], bufs[3][:m]
    return out


def extend_query_multi(trees, sphere_sets, points, ranges, robot_radius, flags=0, capacity=4096):
    """extend_query for n independent instances (trees[i], sphere_sets[i], points[i], ranges[i]) in one launch and
    one host wait; returns one ExtendResult per instance, equal to what extend_query returns for it."""
    n = len(trees)
    if n == 0:
        return []
    d = trees[0].d
    pts = A.as_f64(points, d)
    rr = A.as_f64(ranges).reshape(-1)
    assert len(sphere_sets) == n and pts.shape[0] == n and rr.size == n
    th = (A.vp * n)(*[None if t is None else t.h for t in trees])
    sh = (A.vp * n)(*[None if s is None else s.h for s in sphere_sets])
    ni, nd = np.empty(n, dtype=np.int32), np.empty(n, dtype=np.float64)
    pc, ce, cnt = np.empty(n, dtype=np.uint8), np.empty(n, dtype=np.float64), np.empty(n, dtype=np.int32)
    w = n * capacity
    idx, dist = np.empty(max(w, 1), dtype=np.int32), np.empty(max(w, 1), dtype=np.float64)
    fwd, rev = np.empty(max(w, 1), dtype=np.uint8), np.empty(max(w, 1), dtype=np.uint8)
    L = trees[0].L
    ctx_h = next((t.ctx.h for t in trees if t is not None), None)
    A.check(L.rrtqx_extend_query_multi(th, sh, n, A.ptr(pts), A.ptr(rr), float(robot_radius), int(flags), int(capacity),
                                       A.ptr(ni), A.ptr(nd), A.ptr(pc), A.ptr(ce), A.ptr(cnt), A.ptr(idx), A.ptr(dist),
                                       A.ptr(fwd), A.ptr(rev)), ctx_h)
    outs = []
    for i in range(n):
        out = ExtendResult()
        out.nearest_idx, out.nearest_dist = int(ni[i]), float(nd[i])
        out.point_collides, out.point_cert, out.count = bool(pc[i]), float(ce[i]), int(cnt[i])
        a, b = i * capacity, i * capacity + min(out.count, capacity)
        out.idx, out.dist, out.fwd, out.rev = idx[a:b], dist[a:b], fwd[a:b], rev[a:b]
        outs.append(out)
    return outs


def insert_multi(trees, positions):
    """rrtqx_tree_insert of positions[i] into trees[i] for every i in one asynchronous launch; returns the indices."""
    n = len(trees)
    if n == 0:
        return np.empty(0, dtype=np.int32)
    pos = A.as_f64(positions, trees[0].d)
    assert pos.shape[0] == n
    th = (A.vp * n)(*[None if t is None else t.h for t in trees])
    out = np.empty(n, dtype=np.int32)
    ctx_h = next((t.ctx.h for t in trees if t is not None), None)
    A.check(trees[0].L.rrtqx_tree_insert_multi(th, n, A.ptr(pos), A.ptr(out)), ctx_h)
    return out


class PolygonSet:
    """rrtqx_polygons: the 2-D obstacle list of the Otte generation (kinds 1 = ball, 3 = polygon)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self.L = ctx.L
        h = A.vp()
        A.check(self.L.rrtqx_polygons_create(ctx.h, C.byref(h)), ctx.h)
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.rrtqx_polygons_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def polygon_bound(poly):
        """Bounding circle exactly as the Obstacle(kind, polygon) constructor computes it
        (DRRT_data_structures.jl:229-241): bbox midpoint, radius = sqrt(max_i |v_i - c|^2)."""
        poly = np.asarray(poly, dtype=np.float64).reshape(-1, 2)
        cx = (poly[:, 0].max() + poly[:, 0].min()) / 2.0
        cy = (poly[:, 1].max() + poly[:, 1].min()) / 2.0
        dx, dy = poly[:, 0] - cx, poly[:, 1] - cy
        return cx, cy, float(np.sqrt((dx * dx + dy * dy).max()))

    def upload(self, obstacles, active=None):
        """obstacles: list of ("ball", (cx, cy), r) or ("polygon", vertices Px2)."""
        n = len(obstacles)
        kind = np.zeros(n, dtype=np.int32)
        centers = np.zeros((n, 2))
        radii = np.zeros(n)
        vptr = np.zeros(n + 1, dtype=np.int64)
        verts = []
        for i, ob in enumerate(obstacles):
            if ob[0] == "ball":
                kind[i] = 1
                centers[i] = ob[1]
                radii[i] = ob[2]
            else:
                kind[i] = 3
                v = np.asarray(ob[1], dtype=np.float64).reshape(-1, 2)
                centers[i, 0], centers[i, 1], radii[i] = self.polygon_bound(v)
                verts.append(v)
            vptr[i + 1] = vptr[i] + (len(verts[-1]) if kind[i] == 3 else 0)
        vv = np.ascontiguousarray(np.concatenate(verts, axis=0)) if verts else np.zeros((0, 2))
        act = None if active is None else A.as_u8(np.asarray(active).astype(np.uint8))
        A.check(self.L.rrtqx_polygons_upload(self.h, A.ptr(kind), A.ptr(centers), A.ptr(radii), A.ptr(act), A.ptr(vptr),
                                             A.ptr(vv) if len(vv) else None, n), self.ctx.h)
        self.kind, self.centers, self.radii, self.vptr, self.verts = kind, centers, radii, vptr, vv


def segment_check_2d_batch(polys: PolygonSet, starts, ends, radius, flags=0):
    """explicitEdgeCheck2D OR-ed over the obstacle list for n 2-D segments."""
    starts, ends = A.as_f64(starts, 2), A.as_f64(ends, 2)
    n = starts.shape[0]
    out = np.empty(n, dtype=np.uint8)
    A.check(polys.L.rrtqx_segment_check_2d_batch(polys.h, A.ptr(starts), A.ptr(ends), n, float(radius), int(flags),
                                                 A.ptr(out)), polys.ctx.h)
    return out


def dubins_edge_check_batch(polys: PolygonSet, starts, ends, traj_ptr, traj_xy, robot_radius, min_turn_radius, flags=0):
    """Dubins explicitEdgeCheck OR-ed over the obstacle list; trajectories as CSR (traj_ptr, traj_xy)."""
    starts, ends = A.as_f64(starts, 2), A.as_f64(ends, 2)
    traj_ptr = np.ascontiguousarray(traj_ptr, dtype=np.int64)
    traj_xy = A.as_f64(traj_xy, 2)
    n = starts.shape[0]
    out = np.empty(n, dtype=np.uint8)
    A.check(polys.L.rrtqx_dubins_edge_check_batch(polys.h, A.ptr(starts), A.ptr(ends), A.ptr(traj_ptr),
                                                  A.ptr(traj_xy) if len(traj_xy) else None, n, float(robot_radius),
                                                  float(min_turn_radius), int(flags), A.ptr(out)), polys.ctx.h)
    return out


class DubinsResult:
    """rrtqx_dubins_result: per-edge dist / dubinsType and edge.trajectory[:,1:2] rows as a CSR, device resident."""
    TYPES = ("rsl", "rsr", "rlr", "lsr", "lsl", "lrl")  # edge.dubinsType; -1 is the reference's "xxx"

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self.L = ctx.L
        self.h = A.vp()

    def close(self):
        if getattr(self, "h", None):
            self.L.rrtqx_dubins_result_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sizes(self):
        ne, nr = A.i64(), A.i64()
        A.check(self.L.rrtqx_dubins_result_sizes(self.h, C.byref(ne), C.byref(nr)), self.ctx.h)
        return ne.value, nr.value

    def fetch(self):
        """(dist[n], type[n], traj_ptr[n+1], traj_xy[rows, 2]) as numpy arrays."""
        ne, nr = self.sizes()
        dist = np.empty(ne, dtype=np.float64)
        typ = np.empty(ne, dtype=np.int32)
        ptr = np.zeros(ne + 1, dtype=np.int64)
        xy = np.empty((nr, 2), dtype=np.float64)
        A.check(self.L.rrtqx_dubins_result_fetch(self.h, A.ptr(dist), A.ptr(typ), A.ptr(ptr), A.ptr(xy) if nr else None),
                self.ctx.h)
        return dist, typ, ptr, xy

    def device_pointers(self):
        d, t, p, x = A.vp(), A.vp(), A.vp(), A.vp()
        A.check(self.L.rrtqx_dubins_result_device(self.h, C.byref(d), C.byref(t), C.byref(p), C.byref(x)), self.ctx.h)
        return d.value, t.value, p.value, x.value


def dubins_trajectory_batch(ctx: Context, starts, goals, min_turn_radius, result: DubinsResult | None = None, n_edges=None):
    """calculateTrajectory(S, edge::DubinsEdge) for a batch: starts / goals are n x 4 rows [x y t theta]
    (numpy, or raw device pointers with n_edges given)."""
    if result is None:
        result = DubinsResult(ctx)
    if isinstance(starts, (int, np.integer)):
        n, ps, pg = int(n_edges), int(starts), int(goals)
    else:
        starts, goals = A.as_f64(starts, 4), A.as_f64(goals, 4)
        n, ps, pg = starts.shape[0], A.ptr(starts), A.ptr(goals)
    A.check(ctx.L.rrtqx_dubins_trajectory_batch(ctx.h, ps, pg, n, float(min_turn_radius), C.byref(result.h)), ctx.h)
    return result


def dubins_saturate_batch(ctx: Context, new_points, closest, delta):
    """saturate(newPoint, closestPoint, delta), DubinsEdge version, in place on a copy; returns the n x 4 array."""
    pts = np.array(A.as_f64(new_points, 4), copy=True)
    cl = A.as_f64(closest, 4)
    A.check(ctx.L.rrtqx_dubins_saturate_batch(ctx.h, A.ptr(pts), A.ptr(cl), pts.shape[0], float(delta)), ctx.h)
    return pts


class ExtendDubinsResult:
    """Outputs of one rrtqx_extend_query_dubins call.  Edge 2i runs new -> idx[i], edge 2i+1 idx[i] -> new."""
    __slots__ = ("point", "nearest_idx", "nearest_dist", "count", "idx", "dist", "edge_dist", "edge_type",
                 "edge_collide", "trajectories", "first_edge")


def extend_query_dubins(tree: DeviceTree, polys: PolygonSet, point, r, robot_radius, min_turn_radius, delta=0.0,
                        flags=0, capacity=8192, trajectories: DubinsResult | bool | None = None):
    """The DubinsEdge planner's per-iteration work in one call on the [x y t theta] tree with the theta wrap:
    nearest, saturate (flags | EXTEND_SATURATE), the ball of radius r, and calculateTrajectory + explicitEdgeCheck
    of both edges per neighbour.  trajectories: a DubinsResult to keep the rows in (True: a new one), or None."""
    p = np.array(A.as_f64(point).reshape(-1), copy=True)
    assert p.size == 4, "point must hold [x y t theta]"
    idx, dist = np.empty(max(capacity, 1), dtype=np.int32), np.empty(max(capacity, 1))
    edist, etype = np.empty(2 * max(capacity, 1)), np.empty(2 * max(capacity, 1), dtype=np.int32)
    ecol = np.empty(2 * max(capacity, 1), dtype=np.uint8)
    if trajectories is True:
        trajectories = DubinsResult(tree.ctx)
    ni, nd, cnt = A.i32(0), A.f64(0.0), A.i32(0)
    A.check(tree.L.rrtqx_extend_query_dubins(tree.h, polys.h, A.ptr(p), float(delta), float(r), float(robot_radius),
                                             float(min_turn_radius), int(flags), int(capacity), C.byref(ni),
                                             C.byref(nd), C.byref(cnt), A.ptr(idx), A.ptr(dist), A.ptr(edist),
                                             A.ptr(etype), A.ptr(ecol),
                                             C.byref(trajectories.h) if trajectories is not None else None),
            tree.ctx.h)
    out = ExtendDubinsResult()
    out.point, out.nearest_idx, out.nearest_dist, out.count = p, int(ni.value), float(nd.value), int(cnt.value)
    m = min(out.count, capacity)
    out.idx, out.dist = idx[:m], dist[:m]
    out.edge_dist, out.edge_type, out.edge_collide = edist[:2 * m], etype[:2 * m], ecol[:2 * m]
    out.trajectories, out.first_edge = trajectories, 0
    return out


def extend_query_dubins_multi(trees, poly_sets, points, ranges, robot_radius, min_turn_radius, delta=0.0, flags=0,
                              capacity=1024, trajectories: DubinsResult | bool | None = None):
    """extend_query_dubins for n independent instances (trees[i], poly_sets[i], points[i], ranges[i]) in one call;
    returns one ExtendDubinsResult per instance, equal to what extend_query_dubins returns for it.  The instances
    share one trajectory result: instance i's edges start at its first_edge in the packed edge order."""
    n = len(trees)
    if n == 0:
        return []
    pts = np.array(A.as_f64(points, 4), copy=True)
    rr = A.as_f64(ranges).reshape(-1)
    assert len(poly_sets) == n and pts.shape[0] == n and rr.size == n
    th = (A.vp * n)(*[None if t is None else t.h for t in trees])
    ph = (A.vp * n)(*[None if p is None else p.h for p in poly_sets])
    ni, nd, cnt = np.empty(n, dtype=np.int32), np.empty(n), np.empty(n, dtype=np.int32)
    w = max(n * capacity, 1)
    idx, dist = np.empty(w, dtype=np.int32), np.empty(w)
    edist, etype, ecol = np.empty(2 * w), np.empty(2 * w, dtype=np.int32), np.empty(2 * w, dtype=np.uint8)
    ctx = next((t.ctx for t in trees if t is not None), None)
    if trajectories is True:
        trajectories = DubinsResult(ctx)
    L = ctx.L if ctx is not None else A.lib()
    A.check(L.rrtqx_extend_query_dubins_multi(
        th, ph, n, A.ptr(pts), A.ptr(rr), float(delta), float(robot_radius), float(min_turn_radius), int(flags),
        int(capacity), A.ptr(ni), A.ptr(nd), A.ptr(cnt), A.ptr(idx), A.ptr(dist), A.ptr(edist), A.ptr(etype),
        A.ptr(ecol), C.byref(trajectories.h) if trajectories is not None else None), ctx.h if ctx else None)
    outs, first = [], 0
    for i in range(n):
        out = ExtendDubinsResult()
        out.point, out.nearest_idx, out.nearest_dist, out.count = pts[i], int(ni[i]), float(nd[i]), int(cnt[i])
        m = min(out.count, capacity)
        a, e = i * capacity, 2 * i * capacity
        out.idx, out.dist = idx[a:a + m], dist[a:a + m]
        out.edge_dist, out.edge_type, out.edge_collide = edist[e:e + 2 * m], etype[e:e + 2 * m], ecol[e:e + 2 * m]
        out.trajectories, out.first_edge = trajectories, first
        first += 2 * m
        outs.append(out)
    return outs


def extend_query_dubins_composed(tree: DeviceTree, polys: PolygonSet, point, r, robot_radius, min_turn_radius,
                                 node_positions, delta=0.0, flags=0, trajectories: DubinsResult | None = None,
                                 range_result: RangeResult | None = None):
    """The work of extend_query_dubins through the batch entry points, one blocking call each: nearest ->
    saturate -> range query -> Dubins trajectories -> Dubins edge check (the rows stay on the device).
    node_positions: the caller's host copy of the tree's n x 4 positions (the planner's node table)."""
    p = np.array(A.as_f64(point, 4), copy=True)
    ni, nd = tree.nearest(p)
    if flags & A.EXTEND_SATURATE:
        p = dubins_saturate_batch(tree.ctx, p, node_positions[int(ni[0])], delta)
    res, total = tree.range_query(p, r, want_dist=True, result=range_result)
    idx, dist = res.fetch()
    nb = node_positions[idx]
    starts, goals = np.empty((2 * total, 4)), np.empty((2 * total, 4))
    starts[0::2], starts[1::2] = p, nb          # edge 2i: new -> nbr i, edge 2i+1: nbr i -> new
    goals[0::2], goals[1::2] = nb, p
    if trajectories is None:
        trajectories = DubinsResult(tree.ctx)
    out = ExtendDubinsResult()
    out.point, out.nearest_idx, out.nearest_dist, out.count = p.reshape(-1), int(ni[0]), float(nd[0]), int(total)
    out.idx, out.dist = idx, dist
    out.edge_dist, out.edge_type = np.empty(2 * total), np.empty(2 * total, dtype=np.int32)
    out.edge_collide = np.zeros(2 * total, dtype=np.uint8)
    out.trajectories = trajectories
    dubins_trajectory_batch(tree.ctx, starts, goals, min_turn_radius, result=trajectories)
    if total:
        A.check(tree.L.rrtqx_dubins_result_fetch(trajectories.h, A.ptr(out.edge_dist), A.ptr(out.edge_type), None,
                                                 None), tree.ctx.h)
        _, _, dptr, dxy = trajectories.device_pointers()
        s2, g2 = np.ascontiguousarray(starts[:, :2]), np.ascontiguousarray(goals[:, :2])
        A.check(polys.L.rrtqx_dubins_edge_check_batch(polys.h, A.ptr(s2), A.ptr(g2), dptr, dxy, 2 * total,
                                                      float(robot_radius), float(min_turn_radius), int(flags),
                                                      A.ptr(out.edge_collide)), polys.ctx.h)
    return out


class Comm:
    """rrtqx_comm: the ranks of a sharded job.  Comm.local(ctxs): ONE process driving one context per device (the
    reference's host is one process); Comm.rank(ctx, id, rank, n): one process per GPU (torchrun), `id` being the
    128 bytes rank 0 got from Comm.unique_id() and handed to the others."""

    def __init__(self, h, ctxs):
        self.h, self.ctxs, self.L = h, list(ctxs), ctxs[0].L

    @classmethod
    def local(cls, ctxs):
        arr = (A.vp * len(ctxs))(*[c.h for c in ctxs])
        h = A.vp()
        A.check(ctxs[0].L.rrtqx_comm_init_local(arr, len(ctxs), C.byref(h)), ctxs[0].h)
        return cls(h, ctxs)

    @staticmethod
    def unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        A.check(A.lib().rrtqx_comm_unique_id(buf), None)
        return buf.raw

    @classmethod
    def rank(cls, ctx, unique_id: bytes, rank: int, n_ranks: int):
        h = A.vp()
        buf = C.create_string_buffer(bytes(unique_id), 128)
        A.check(ctx.L.rrtqx_comm_init_rank(ctx.h, buf, int(rank), int(n_ranks), C.byref(h)), ctx.h)
        return cls(h, [ctx])

    def close(self):
        if getattr(self, "h", None):
            self.L.rrtqx_comm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self):
        v = [A.i32(0) for _ in range(5)]
        A.check(self.L.rrtqx_comm_info(self.h, *[C.byref(x) for x in v]), self.ctxs[0].h)
        return {"n_ranks": v[0].value, "n_local": v[1].value, "first_rank": v[2].value,
                "peer_stores": bool(v[3].value), "nccl_version": v[4].value}

    def packed_words(self, n_edges: int):
        a, b = A.i64(0), A.i64(0)
        A.check(self.L.rrtqx_comm_packed_words(self.h, int(n_edges), C.byref(a), C.byref(b)), self.ctxs[0].h)
        return int(a.value), int(b.value)

    def allgather(self, send_ptrs, recv_ptrs, bytes_per_rank: int, side_stream: bool = False):
        """send_ptrs / recv_ptrs: one device pointer per local rank."""
        n = len(self.ctxs)
        s = (A.vp * n)(*[A.ptr(p) for p in send_ptrs])
        r = (A.vp * n)(*[A.ptr(p) for p in recv_ptrs])
        A.check(self.L.rrtqx_comm_allgather(self.h, s, r, int(bytes_per_rank), 1 if side_stream else 0), self.ctxs[0].h)

    def join(self):
        A.check(self.L.rrtqx_comm_join(self.h), self.ctxs[0].h)

    def edge_check_sharded(self, trees, spheres, src_ptrs, dst_ptrs, n_edges, robot_radius, packed_ptrs, flags=0):
        """explicitEdgeCheck of one replicated edge list, sharded over the ranks; every rank's packed_ptrs[i] (device,
        packed_words(n_edges)[0] uint32 words) receives ALL flags: edge e = bit e % 32 of word e // 32."""
        n = len(self.ctxs)
        t = (A.vp * n)(*[x.h for x in trees])
        sp = (A.vp * n)(*[x.h for x in spheres])
        s = (A.vp * n)(*[A.ptr(p) for p in src_ptrs])
        d = (A.vp * n)(*[A.ptr(p) for p in dst_ptrs])
        o = (A.vp * n)(*[A.ptr(p) for p in packed_ptrs])
        A.check(self.L.rrtqx_edge_check_batch_sharded(self.h, t, sp, s, d, int(n_edges), float(robot_radius), int(flags), o),
                self.ctxs[0].h)


def unpack_flags(words, n_edges: int) -> np.ndarray:
    """Bit-packed flags of Comm.edge_check_sharded (host uint32 array) -> uint8[n_edges]."""
    w = np.ascontiguousarray(words, dtype=np.uint32)
    return np.unpackbits(w.view(np.uint8), bitorder="little")[:n_edges]
