#!/usr/bin/env python
"""bench.py -- headline benchmark of the RRTQX_3D geometric hot path on B200.

Metric (BASELINE.json): kd range queries/s on a 1M-node 3-D tree (config C2: 1M
kdFindWithinRange queries at the RRTx shrinking-ball radius, neighbour indices AND
distance keys produced), plus edge collision checks/s for the obstacle-add sweep
(config C3) as an extra object on the same JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One process per GPU (torchrun for N > 1): the tree is replicated, every rank owns its
own batch of queries (weak scaling, no data-path collective; per-query counts are
all-gathered over NCCL as the fixed-size result gather).  Prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from rrtqx_3d_b200 import workloads as W  # noqa: E402

# the kernel the library launches for C2 (RRTQX_RANGE_KERNEL=4 selects the previous generation for A/B runs)
DOMINANT_KERNEL = ("range_fused_kernel<3,2,28,576>" if os.environ.get("RRTQX_RANGE_KERNEL") == "4"
                   else "range_v5_kernel<3,24,704,256,uniform>")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed ncu capture
    (profiles/range_traffic.json, written by scripts/write_traffic.py from the same `ncu --set full` report as the
    committed profile summary)."""
    p = os.path.join(ROOT, "profiles", "range_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("dram_bytes_per_launch")
    return None


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for k, nm in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_range_baseline(pts, qs, r, seconds_target=12.0, nthreads=None):
    """Oracle (CPU restatement of the reference kd tree) on a bounded sample of the workload."""
    import oracle
    nthreads = nthreads or os.cpu_count() or 1
    t0 = time.perf_counter()
    tree = oracle.KDTree(3)
    tree.insert_batch(pts)
    build_s = time.perf_counter() - t0
    probe = min(len(qs), 64 * nthreads)
    t0 = time.perf_counter()
    tree.range_batch(r, qs[:probe], want_lists=True, nthreads=nthreads)
    dt = time.perf_counter() - t0
    rate = probe / dt
    sample = int(min(len(qs), max(probe, rate * seconds_target)))
    t0 = time.perf_counter()
    counts, offsets, idx, key = tree.range_batch(r, qs[:sample], want_lists=True, nthreads=nthreads)
    dt = time.perf_counter() - t0
    return {"value": sample / dt, "unit": "queries/s", "cores": nthreads, "kind": "port",
            "sample": f"first {sample} of {len(qs)} C2 queries (idx+key lists), oracle kd tree of {len(pts)} nodes "
                      f"built in {build_s:.1f}s, {dt:.1f}s timed",
            "mean_neighbours": float(counts.mean())}, tree


def julia_reference_rate(pts, qs, r, seconds=20.0):
    """The REAL reference (Julia) on a sample of the workload, when a `julia` binary and the reference tree
    (RRTQX_REFERENCE_DIR=<...>/code_RRTQx_3D) are present; None otherwise.  Single-threaded, like the reference."""
    import shutil
    import subprocess
    import tempfile
    ref = os.environ.get("RRTQX_REFERENCE_DIR")
    if not shutil.which("julia") or not ref or not os.path.isdir(ref):
        return None
    here = os.path.dirname(os.path.abspath(__file__))
    with tempfile.TemporaryDirectory() as td:
        fp, fq = os.path.join(td, "p.f64"), os.path.join(td, "q.f64")
        np.ascontiguousarray(pts, dtype=np.float64).tofile(fp)
        nq = min(len(qs), 20000)
        np.ascontiguousarray(qs[:nq], dtype=np.float64).tofile(fq)
        try:
            out = subprocess.run(["julia", os.path.join(here, "julia", "bench_reference.jl"), ref, fp, fq, str(len(pts)),
                                  str(nq), repr(float(r)), str(seconds)], capture_output=True, text=True, timeout=1800).stdout
            kv = dict(t.split("=") for t in out.strip().split() if "=" in t)
            return {"value": float(kv["queries_per_s"]), "unit": "queries/s", "cores": 1, "kind": "reference",
                    "sample": f"{kv['queries']} C2 queries through the reference's kdFindWithinRange (Julia, 1 thread)"}
        except Exception as exc:  # a broken Julia installation must not take the bench down
            return {"error": repr(exc)}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU algorithm -- the Julia reference itself when `julia` and
    RRTQX_REFERENCE_DIR are present (julia/bench_reference.jl), else the oracle port (no Julia in this image)."""
    if rank != 0:
        return
    nthreads = os.cpu_count() or 1
    pts, qs, r = W.c2_workload(args.nodes, args.queries)
    jl = julia_reference_rate(pts, qs, r)
    if jl and "value" in jl:
        line = {"impl": "reference", "metric": "kd_range_queries_per_s", "value": jl["value"], "unit": "queries/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": None,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "C2 batched neighbour sweep: 1M-node uniform 3-D tree, kdFindWithinRange at the RRTx "
                                       "shrinking-ball radius, idx + distance keys", "nodes": args.nodes,
                           "queries_per_gpu": args.queries, "radius": r, "cpu_arm": jl["sample"]},
                "cpu_baseline": jl,
                "e2e": {"value": jl["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return
    import oracle
    tree = oracle.KDTree(3)
    tree.insert_batch(pts)
    probe = min(len(qs), 64 * nthreads)
    t0 = time.perf_counter()
    tree.range_batch(r, qs[:probe], nthreads=nthreads)
    rate = probe / (time.perf_counter() - t0)
    budget_s = 120.0 / max(1, args.steps + args.warmup)      # whole run within a few minutes
    sample = int(min(len(qs), max(nthreads, rate * min(budget_s, 15.0))))
    times = []
    for it in range(args.warmup + args.steps):
        lo = (it * sample) % max(1, len(qs) - sample + 1)
        t0 = time.perf_counter()
        tree.range_batch(r, qs[lo:lo + sample], nthreads=nthreads)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = sample / (ms / 1e3)
    line = {"impl": "reference", "metric": "kd_range_queries_per_s", "value": value, "unit": "queries/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C2 batched neighbour sweep: 1M-node uniform 3-D tree, kdFindWithinRange at the RRTx "
                                   "shrinking-ball radius, idx + distance keys",
                       "nodes": args.nodes, "queries_per_gpu": args.queries, "radius": r,
                       "cpu_arm": f"each step is a bounded sample of {sample} queries of the workload (all host threads)"},
            "cpu_baseline": {"value": value, "unit": "queries/s", "cores": nthreads, "kind": "port",
                             "sample": f"{sample} C2 queries per step (oracle port of kdFindWithinRange, pthreads)"},
            "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def tensor_from_ptr(torch_mod, p, n, dtype):
    # zero-copy view of library-owned device memory through the CUDA array interface
    class _Holder:
        pass
    h = _Holder()
    typestr = {torch_mod.int32: "<i4", torch_mod.float64: "<f8"}[dtype]
    h.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (int(p), False), "version": 3}
    return torch_mod.as_tensor(h, device="cuda")


DUMP_MAX_BYTES = 64 << 20
DUMP_COUNT_QUERIES = 1 << 20     # counts of all queries at the default size
DUMP_LIST_QUERIES = 4096         # ~1.8M neighbours at the default radius
DUMP_SEED = 77


def dump_range_outputs(out_dir, res, n_queries):
    """--dump-outputs: what the caller of the timed C2 step receives, from the result of the LAST timed step, as
    float64 .npy files under out_dir (at most DUMP_MAX_BYTES).  Queries are sampled with a fixed splitmix64 seed:
      query_index.npy        ascending indices of up to DUMP_COUNT_QUERIES queries (all of them at the default size)
      counts.npy             their neighbour counts
      list_query_index.npy   ascending indices of up to DUMP_LIST_QUERIES of those queries (fewer if the lists would
                             exceed the size limit)
      neighbour_idx.npy      their neighbour lists, concatenated in that order, each list in ascending node index
      neighbour_dist.npy     the distance key of each of those neighbours
    A list is a set (include/rrtqx_b200.h): its order on the device and the offsets that place it in memory are not
    part of the result, so they are not written and two builds compare file for file."""
    import torch
    counts, offsets = res.layout()
    order = np.argsort(W.splitmix64(DUMP_SEED, 0, n_queries), kind="stable")
    sel = np.sort(order[:min(n_queries, DUMP_COUNT_QUERIES)])
    take = order[:min(n_queries, DUMP_LIST_QUERIES)]
    room = DUMP_MAX_BYTES - 16 * len(sel) - 4096          # 4096: the five .npy headers
    take = np.sort(take[:np.searchsorted(np.cumsum(16 * counts[take].astype(np.int64) + 8), room, side="right")])
    n = counts[take].astype(np.int64)
    owner = np.repeat(np.arange(len(take)), n)
    pos = offsets[take][owner] + (np.arange(int(n.sum())) - np.repeat(np.cumsum(n) - n, n))
    _, _, idx_p, dist_p = res.device_pointers()
    total = res.sizes()[1]
    pos_d = torch.from_numpy(pos).cuda()
    idx = tensor_from_ptr(torch, idx_p, total, torch.int32)[pos_d].cpu().numpy()
    dist = tensor_from_ptr(torch, dist_p, total, torch.float64)[pos_d].cpu().numpy()
    by_node = np.lexsort((idx, owner))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("query_index", sel), ("counts", counts[sel]), ("list_query_index", take),
                    ("neighbour_idx", idx[by_node]), ("neighbour_dist", dist[by_node])):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


_C3_CACHE = {}


def build_c3_edges(tree, pts, r_edge):
    """Memoised per process (the sweep and the C5 leg use the same edge set)."""
    key = (id(tree), float(r_edge))
    if key not in _C3_CACHE:
        _C3_CACHE[key] = _build_c3_edges(tree, pts, r_edge)
    return _C3_CACHE[key]


def _build_c3_edges(tree, pts, r_edge):
    """C3 edge set: all ordered pairs (i, j), i != j, within r_edge, generated with the range kernel;
    parent[i] = lowest-index neighbour below i, else the node's kd parent (always a lower index)."""
    res, total = tree.range_query(pts, r_edge, want_dist=False)
    counts, offsets = res.layout()
    idx, _ = res.fetch(want_dist=False)
    order = np.argsort(offsets, kind="stable")
    src = np.empty(total, dtype=np.int32)
    src[:] = np.repeat(order.astype(np.int32), counts[order])     # lists are packed in offset order
    keep = src != idx
    src, dst = src[keep], idx[keep]
    # canonical order (the kernel's list order depends on its atomics): every rank shards the SAME array
    order = np.argsort(src.astype(np.int64) << 32 | dst.astype(np.int64), kind="stable")
    src, dst = np.ascontiguousarray(src[order]), np.ascontiguousarray(dst[order])
    parent = tree.kd_fields()[0].copy()
    lower = dst < src
    cand = np.full(len(pts), np.iinfo(np.int32).max, dtype=np.int32)
    np.minimum.at(cand, src[lower], dst[lower])
    has = cand != np.iinfo(np.int32).max
    parent[has] = cand[has]
    res.close()
    return src, dst, parent


def c1_replay(ctx, n_iter):
    """Config C1: planner-style incremental loop (one sample per iteration) through rrtqx_extend_query +
    rrtqx_tree_insert on the GPU, and the same geometric work through the oracle on the CPU (every 25th
    iteration timed, trees kept identical)."""
    import ctypes as C

    import oracle
    from rrtqx_3d_b200 import _abi as A
    from rrtqx_3d_b200.device import DeviceTree, SphereSet, extend_query
    centers, radii, _ = W.building2_spheres()
    S = SphereSet(ctx, centers, radii)
    samples = W.uniform_points(1, n_iter, [-W.ENV_RAD] * 3, [W.ENV_RAD] * 3)
    goal = np.array([4.0, 16.5, -7.5])
    t = DeviceTree(ctx, 3)
    t.insert(goal)
    accept = np.zeros(n_iter, dtype=bool)
    bufs = (np.empty(8192, np.int32), np.empty(8192, np.float64), np.empty(8192, np.uint8), np.empty(8192, np.uint8))
    n = 1
    nbrs = 0
    t0 = time.perf_counter()
    for it in range(n_iter):
        r = W.shrinking_ball_radius(n, 3, W.DELTA, W.BALL_CONSTANT)
        res = extend_query(t, S, samples[it], r, W.ROBOT_RADIUS, A.CHECK_QUICK_PASS, capacity=8192, bufs=bufs)
        nbrs += res.count
        if not res.point_collides:
            t.insert(samples[it])
            accept[it] = True
            n += 1
    gpu_s = time.perf_counter() - t0
    # CPU: same sequence, geometric work of every 25th iteration timed
    L = oracle.lib()
    sph, ns = oracle.make_spheres(centers, radii)
    orc = oracle.KDTree(3)
    orc.insert(goal)
    P = lambda a: oracle._p(np.ascontiguousarray(a, dtype=np.float64), oracle.c_f64p)
    cpu_s, cpu_n = 0.0, 0
    c = C.c_double()
    for it in range(n_iter):
        if it % 25 == 0:
            p = samples[it]
            pos = None
            t1 = time.perf_counter()
            r = W.shrinking_ball_radius(len(orc), 3, W.DELTA, W.BALL_CONSTANT)
            orc.find_nearest(p)
            L.orc_point_check(sph, ns, 0, P(p), W.ROBOT_RADIUS, C.byref(c))
            idx, key = orc.find_within_range(r, p)
            orc.empty(idx)
            k = len(idx)
            if k:
                src = np.full(2 * k, len(orc), dtype=np.int32)       # virtual node index of the new sample
                dst = np.concatenate([idx, idx]).astype(np.int32)
                src[k:], dst[k:] = idx, len(orc)
                ptr = L.orc_kd_positions
                ptr.restype = C.POINTER(C.c_double)
                ptr.argtypes = [C.c_void_p]
                pos = np.concatenate([np.ctypeslib.as_array(ptr(orc.h), shape=(len(orc), 3)), p.reshape(1, 3)])
                out = np.zeros(2 * k, dtype=np.uint8)
                L.orc_edge_check_batch(sph, ns, P(pos), 3, oracle._p(src, oracle.c_i32p), oracle._p(dst, oracle.c_i32p), 0,
                                       2 * k, W.ROBOT_RADIUS, 0, oracle._p(out, oracle.c_u8p), 1)
            cpu_s += time.perf_counter() - t1
            cpu_n += 1
        if accept[it]:
            orc.insert(samples[it])
    return {"workload": "C1 RRTx SimpleEdge 3-D replay: per iteration nearest + node check + range(r(n)) + 2k edge checks "
                        "(31 building2 spheres) + insert",
            "iterations": n_iter, "nodes_final": n, "mean_neighbours": nbrs / n_iter,
            "gpu_us_per_iteration": 1e6 * gpu_s / n_iter, "cpu_us_per_iteration": 1e6 * cpu_s / max(cpu_n, 1),
            "cpu": "oracle, 1 thread (the reference planner is single-threaded), every 25th iteration timed",
            "note": "latency-bound: one launch + one stream synchronise per iteration, results via mapped pinned memory"}


def c4_dubins(ctx, n_edges, steps):
    """Config C4: Dubins edges between poses in [-50,50]^2 x [0,2pi): the six-word solver + trajectory
    discretisation on the device, then the sampled-trajectory collision check against 100 city-block polygons,
    trajectories never leaving the GPU.  CPU: the oracle's solver + check on a bounded sample, one thread."""
    import ctypes as C

    import oracle
    import torch
    from rrtqx_3d_b200 import _abi as A
    from rrtqx_3d_b200.device import DubinsResult, PolygonSet, dubins_trajectory_batch
    u = W.uniform01(44, 0, 6 * n_edges).reshape(n_edges, 6)
    s = np.zeros((n_edges, 4))
    s[:, 0], s[:, 1], s[:, 3] = -50 + 100 * u[:, 0], -50 + 100 * u[:, 1], 2 * np.pi * u[:, 2]
    ang, rad = 2 * np.pi * u[:, 3], 4.0 * np.sqrt(u[:, 4])
    g = np.zeros((n_edges, 4))
    g[:, 0], g[:, 1], g[:, 3] = s[:, 0] + rad * np.cos(ang), s[:, 1] + rad * np.sin(ang), 2 * np.pi * u[:, 5]
    P = PolygonSet(ctx)
    P.upload(W.c4_city_blocks())
    ds, dg = torch.from_numpy(s).cuda(), torch.from_numpy(g).cuda()
    s2, g2 = torch.from_numpy(np.ascontiguousarray(s[:, :2])).cuda(), torch.from_numpy(np.ascontiguousarray(g[:, :2])).cuda()
    out = torch.empty(n_edges, dtype=torch.uint8, device="cuda")
    res = DubinsResult(ctx)
    t_solve, t_check = [], []
    for it in range(3 + steps):
        dubins_trajectory_batch(ctx, ds.data_ptr(), dg.data_ptr(), 1.0, result=res, n_edges=n_edges)
        _, _, dptr, dxy = res.device_pointers()
        A.check(ctx.L.rrtqx_dubins_edge_check_batch(P.h, s2.data_ptr(), g2.data_ptr(), dptr, dxy, n_edges, 0.5, 1.0, 0,
                                                    out.data_ptr()), ctx.h)
        if it >= 3:
            t_solve.append(ctx.last_phase_ms("dubins_solve") + ctx.last_phase_ms("dubins_emit"))
            t_check.append(ctx.last_phase_ms("dubins_check"))
    _, rows = res.sizes()
    ms_s, ms_c = float(np.mean(t_solve)), float(np.mean(t_check))
    # the kd side of C4: 200k nodes in [-50,50]^2 x {0} x [0,2pi), 4-D Euclid with the theta ghost identity
    # (KDTree{T}(4, KDdist, [4], [2pi]), DRRT.jl:3312), 200k range queries at a radius giving E[k] ~ 16
    import math
    from rrtqx_3d_b200.device import DeviceTree, RangeResult
    lo4, hi4 = [-50.0, -50.0, 0.0, 0.0], [50.0, 50.0, 0.0, 2.0 * math.pi]
    nodes4 = W.uniform_points(4, 200_000, lo4, hi4)
    q4 = torch.from_numpy(W.uniform_points(5, 200_000, lo4, hi4)).cuda()
    t4 = DeviceTree(ctx, 4, wraps=[3], wrap_points=[2.0 * math.pi])
    t4.insert_batch(nodes4)
    r4res = RangeResult(ctx)
    kd_ms = []
    for it in range(3 + steps):
        _, k4 = t4.range_query(q4, 1.06, result=r4res, n_queries=200_000)
        if it >= 3:
            kd_ms.append(ctx.last_phase_ms("range_query"))
    kd_ms = float(np.mean(kd_ms))
    # the Otte / Dubins replanning sweep (DRRT.jl:3127-3197) on the C4 graph: every node's neighbours within 1.06 as
    # out-edges, the first neighbour as parent, trajectories of all items solved on the device and kept resident
    from rrtqx_3d_b200.device import EdgeSet, SweepResult
    resn, totn = t4.range_query(nodes4, 1.06, want_dist=False)
    cntn, offn = resn.layout()
    idxn, _ = resn.fetch(want_dist=False)
    by_off = np.argsort(offn, kind="stable")
    srcn = np.repeat(by_off.astype(np.int32), cntn[by_off])
    dstn = idxn[:totn].astype(np.int32)
    keep = srcn != dstn
    srcn, dstn = srcn[keep], dstn[keep]
    o2 = np.argsort(srcn, kind="stable")
    srcn, dstn = np.ascontiguousarray(srcn[o2]), np.ascontiguousarray(dstn[o2])
    par = np.full(len(nodes4), -1, dtype=np.int32)
    first = np.r_[True, srcn[1:] != srcn[:-1]]
    par[srcn[first]] = dstn[first]
    par[0] = -1
    resn.close()
    E4 = EdgeSet(t4)
    E4.upload(srcn, dstn, par)
    ctx.sync()
    t0 = time.perf_counter()
    rows4 = E4.solve_trajectories(1.0)
    ctx.sync()
    solve_all_ms = 1e3 * (time.perf_counter() - t0)
    all_obs = np.arange(len(P.kind), dtype=np.int32)
    sw = SweepResult(ctx)
    sw_ms, one_ms = [], []
    for it in range(3 + steps):
        E4.add_sweep_2d(P, all_obs, 0.5, 5.0, 1.0, result=sw)
        if it >= 3:
            sw_ms.append(ctx.last_phase_ms("add_sweep_2d"))
    blocked4, orphans4 = sw.sizes()[0], sw.sizes()[1]
    for o in range(0, len(all_obs), max(1, len(all_obs) // 8)):
        E4.add_sweep_2d(P, [o], 0.5, 5.0, 1.0, result=sw)
        one_ms.append(ctx.last_phase_ms("add_sweep_2d"))
    sweep_2d = {"nodes": len(nodes4), "edges": int(len(srcn)), "trajectory_rows": int(rows4), "obstacles": int(len(all_obs)),
                "solve_trajectories_ms_wall": solve_all_ms, "ms": float(np.mean(sw_ms)),
                "edges_per_s": len(srcn) / (float(np.mean(sw_ms)) / 1e3), "blocked_edges": int(blocked4),
                "orphans": int(orphans4), "single_obstacle_ms": float(np.median(one_ms)),
                "single_obstacle_ms_each": [round(float(x), 4) for x in one_ms],
                "note": "addNewObstacle of the Otte generation with DubinsEdge: theta-wrapped start-node filter, "
                        "sampled-trajectory check of every out-edge and parent edge of the candidates"}
    sw.close()
    # CPU sample
    L = oracle.lib()
    f = lambda a: oracle._p(np.ascontiguousarray(a, dtype=np.float64), oracle.c_f64p)
    obs = []
    for i in range(len(P.kind)):
        ob = oracle.Obstacle2D()
        ob.kind = int(P.kind[i])
        ob.pos[0], ob.pos[1] = P.centers[i]
        ob.radius, ob.life_span, ob.unused = P.radii[i], float("inf"), 0
        v = np.ascontiguousarray(P.verts[P.vptr[i]:P.vptr[i + 1]])
        ob.n_vert, ob._keep, ob.poly = len(v), v, oracle._p(v, oracle.c_f64p)
        obs.append(ob)
    n_cpu = min(n_edges, 3000)
    t0 = time.perf_counter()
    hits = 0
    for e in range(n_cpu):
        _, _, traj = oracle.dubins_trajectory(s[e], g[e], 1.0)
        for ob in obs:
            if L.orc_edge_check_dubins(C.byref(ob), f(s[e, :2]), f(g[e, :2]), f(traj), len(traj), 0.5, 1.0):
                hits += 1
                break
    cpu_s = time.perf_counter() - t0
    return {"workload": "C4 Dubins edges (r_turn 1, r_robot 0.5) vs 100 city-block polygons: device solver + "
                        "trajectory discretisation + sampled-trajectory collision check",
            "edges": n_edges, "trajectory_rows": rows, "solve_ms": ms_s, "check_ms": ms_c,
            "edges_per_s": n_edges / ((ms_s + ms_c) / 1e3), "colliding_edges": int(out.sum().item()),
            "cpu_edges_per_s": n_cpu / cpu_s, "cpu": f"oracle solver + check, 1 thread, first {n_cpu} edges "
                                                    "(python call overhead included)",
            "algorithmic_bytes": n_edges * (64 + 16 + 1) + rows * 16 * 2,
            "sweep_2d": sweep_2d,
            "kd_wrap_queries": {"nodes": 200_000, "queries": 200_000, "radius": 1.06, "mean_neighbours": k4 / 200_000,
                                "ms": kd_ms, "queries_per_s": 200_000 / (kd_ms / 1e3),
                                "note": "theta ghost identities run as (real, ghost) pairs of the range kernel"}}


def c5_instances(ctx, rank, world, n_instances, n_iter):
    """Config C5a: independent C1-style planning instances (seeds 1..n), round-robin over ranks; each instance is
    the incremental loop extend_query + insert.  Returns (iterations done by this rank, seconds)."""
    from rrtqx_3d_b200 import _abi as A
    from rrtqx_3d_b200.device import DeviceTree, SphereSet, extend_query
    centers, radii, _ = W.building2_spheres()
    S = SphereSet(ctx, centers, radii)
    bufs = (np.empty(8192, np.int32), np.empty(8192, np.float64), np.empty(8192, np.uint8), np.empty(8192, np.uint8))
    done = 0
    t0 = time.perf_counter()
    for inst in range(rank, n_instances, world):
        samples = W.uniform_points(1 + inst, n_iter, [-W.ENV_RAD] * 3, [W.ENV_RAD] * 3)
        t = DeviceTree(ctx, 3)
        t.insert(np.array([4.0, 16.5, -7.5]))
        n = 1
        for it in range(n_iter):
            r = W.shrinking_ball_radius(n, 3, W.DELTA, W.BALL_CONSTANT)
            res = extend_query(t, S, samples[it], r, W.ROBOT_RADIUS, A.CHECK_QUICK_PASS, capacity=8192, bufs=bufs)
            if not res.point_collides:
                t.insert(samples[it])
                n += 1
        done += n_iter
        t.close()
    return done, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nodes", type=int, default=1_000_000)
    ap.add_argument("--queries", type=int, default=1_000_000)
    ap.add_argument("--radius", type=float, default=None)
    ap.add_argument("--occupancy", type=float, default=None)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-count-gather", action="store_true", help="diagnosis: skip the per-step gather of the counts (N > 1)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-c1", action="store_true")
    ap.add_argument("--c1-iterations", type=int, default=20000)
    ap.add_argument("--sweep-edge-radius", type=float, default=0.5346)
    ap.add_argument("--sweep-obstacles", type=int, default=256)
    ap.add_argument("--no-c4", action="store_true")
    ap.add_argument("--c4-edges", type=int, default=200_000)
    ap.add_argument("--no-c5", action="store_true")
    ap.add_argument("--c5-instances", type=int, default=64)
    ap.add_argument("--c5-iterations", type=int, default=1000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed C2 step computed to DIR/<name>.npy (see dump_range_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from rrtqx_3d_b200.device import Comm, Context, DeviceTree, EdgeSet, RangeResult, SphereSet, SweepResult

    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # ONE stream for torch and the library.  torch's default stream has handle 0, which rrtqx_ctx_create reads as "no
    # stream given" (it then creates its own): the flush memsets and the timing events would sit on another stream
    # than the kernels they are meant to bracket.  A non-default torch stream has a real handle.
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    ctx = Context(local_rank, stream.cuda_stream)
    comm = None
    if world > 1:   # the library's own communicator (NCCL inside librrtqx_b200.so); torch only moves the unique id
        uid = [Comm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        comm = Comm.rank(ctx, uid[0], rank, world)
    peak_gbs, peak_src = measured_peaks()

    # ------------------------------------------------------------- workload C2
    pts, _, r = W.c2_workload(args.nodes, 1, radius=args.radius)
    qs = W.uniform_points(2 + rank, args.queries, [-W.ENV_RAD] * 3, [W.ENV_RAD] * 3)   # own batch per rank
    tree = DeviceTree(ctx, 3)
    if args.occupancy:
        tree.set_cell_occupancy(args.occupancy)
    tree.insert_batch(pts)
    dq = torch.from_numpy(qs).cuda()                     # inputs resident in HBM before the timed region
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    res = RangeResult(ctx)
    gathered = torch.empty(world * args.queries, dtype=torch.int32, device="cuda") if world > 1 else None

    counts_view = {}

    def step():
        _, total = tree.range_query(dq, r, want_dist=True, result=res, n_queries=args.queries)
        if world > 1 and not args.no_count_gather:   # fixed-size result gather: per-query counts of every rank (NCCL over NVLink, inside the
            # library, on its side stream: the next step's kernel does not wait for it)
            comm.allgather([res.device_pointers()[0]], [gathered.data_ptr()], args.queries * 4, side_stream=True)
        return total

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        flush.zero_()
        total = step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler.rows.clear()            # keep only samples taken during the timed region
    launches0 = ctx.kernel_launches()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kern = {"range_sort": [], "range_count": [], "range_scan": [], "range_fill": []}
    torch.cuda.synchronize()
    wall0 = time.perf_counter()
    for a, b in ev:
        flush.zero_()                                    # L2 flush between timed iterations (outside the events)
        a.record(stream)
        total = step()
        b.record(stream)
        b.synchronize()
        for k in kern:
            try:
                kern[k].append(ctx.last_phase_ms(k))
            except Exception:
                pass
    tail_ms = 0.0
    if world > 1:   # the gathers still in flight on the side stream belong to the timed steps: wait for them
        t_end = torch.cuda.Event(enable_timing=True)
        comm.join()
        t_end.record(stream)
        torch.cuda.synchronize()
        tail_ms = ev[-1][1].elapsed_time(t_end)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    launches = ctx.kernel_launches() - launches0
    ms_local = float(np.mean([a.elapsed_time(b) for a, b in ev])) + tail_ms / max(1, len(ev))
    if world > 1:
        tmax = torch.tensor([ms_local], device="cuda", dtype=torch.float64)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax.item())
        tot_t = torch.tensor([total], device="cuda", dtype=torch.int64)
        dist.all_reduce(tot_t)
        total_all = int(tot_t.item())
    else:
        ms, total_all = ms_local, total
    value = world * args.queries / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        dump_range_outputs(args.dump_outputs, res, args.queries)

    # roofline of the step: compulsory bytes (SURVEY 8d): N*24 + Q*24 + (Q+1)*8 + K*(4+8)
    K = total
    alg_bytes = args.nodes * 24 + args.queries * 24 + (args.queries + 1) * 8 + K * 12
    kern_ms = {k: float(np.mean(v)) for k, v in kern.items() if v}
    # contract: achieved = algorithmic bytes of one launch of the dominant kernel / its average launch duration,
    # measured live with CUDA events on the launching stream (the library brackets the launch: phase "range_fill").
    # The whole step (query sort + kernel) is reported next to it as step_*.
    fill_ms = kern_ms["range_fill"]
    achieved = alg_bytes / (fill_ms / 1e3) / 1e9
    step_achieved = alg_bytes / (ms_local / 1e3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
                "traffic": ncu_traffic(), "peak_source": peak_src, "algorithmic_bytes_per_step": alg_bytes,
                "note": "achieved = compulsory bytes of the range-query step / CUDA-event duration of the dominant kernel "
                        + DOMINANT_KERNEL + " (one launch per step, events recorded by the library on its stream); "
                        "step_* = the same bytes / the whole step (query sort + kernel)",
                "kernel_ms": kern_ms, "dominant_kernel_share": fill_ms / ms_local,
                "step_achieved": step_achieved, "step_frac": step_achieved / peak_gbs}

    line = {"metric": "kd_range_queries_per_s", "value": value, "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C2 batched neighbour sweep: 1M-node uniform 3-D tree, kdFindWithinRange at the RRTx "
                                   "shrinking-ball radius, idx + distance keys",
                       "nodes": args.nodes, "queries_per_gpu": args.queries, "radius": r,
                       "neighbours_per_step_rank0": K, "mean_neighbours": K / args.queries,
                       "parallelism": f"replicated tree x {world} query shards", "l2_flush_between_steps": True,
                       "l2_flush": "256 MiB memset on the SAME stream as the library's kernels between timed iterations (scripts/exp_flush.py: write, write+read and copy flushes give the same timings)",
                       "count_gather": ("rrtqx_comm_allgather (NCCL inside the library) on the communicator's side stream; "
                                        "the timed steps include the wait for the last gather") if world > 1 else "none (one rank)"},
            "clocks": clocks, "gpu_launches": launches, "roofline": roofline,
            "wall_ms_per_step_incl_flush": 1e3 * wall / args.steps}

    # ------------------------------------------------------- extra: sparse variant (SURVEY 8d): index cost vs output cost
    try:
        sp_r = 0.7795
        sp = []
        res_sp = RangeResult(ctx)
        for it in range(3 + max(3, min(args.steps, 10))):
            flush.zero_()
            _, k_sp = tree.range_query(dq, sp_r, want_dist=True, result=res_sp, n_queries=args.queries)
            if it >= 3:
                sp.append(ctx.last_phase_ms("range_query"))
        sp_ms = float(np.mean(sp))
        sp_bytes = args.nodes * 24 + args.queries * 24 + (args.queries + 1) * 8 + k_sp * 12
        line["sparse_variant"] = {"radius": sp_r, "mean_neighbours": k_sp / args.queries, "ms": sp_ms,
                                  "queries_per_s": args.queries / (sp_ms / 1e3), "algorithmic_bytes": sp_bytes,
                                  "hbm_frac": sp_bytes / (sp_ms / 1e3) / 1e9 / peak_gbs,
                                  "note": "same tree and queries at a radius with ~30 neighbours: set-up + rows dominate"}
        res_sp.close()
    except Exception as exc:
        line["sparse_variant"] = {"error": repr(exc)}

    # ------------------------------------------------------- extra: batched kdFindNearest on the same workload
    try:
        nn_idx = torch.empty(args.queries, dtype=torch.int32, device="cuda")
        nn_dist = torch.empty(args.queries, dtype=torch.float64, device="cuda")
        nts = []
        for it in range(3 + max(3, min(args.steps, 10))):
            flush.zero_()
            tree.nearest(dq.data_ptr(), n_queries=args.queries, idx_out=nn_idx.data_ptr(), dist_out=nn_dist.data_ptr())
            if it >= 3:
                nts.append(ctx.last_phase_ms("nearest"))
        nms = float(np.mean(nts))
        nbytes = args.nodes * 24 + args.queries * 24 + args.queries * 12
        line["nearest"] = {"workload": "kdFindNearest for the same 1M queries (query sort + thread-per-query kernel)",
                           "ms": nms, "queries_per_s": args.queries / (nms / 1e3), "algorithmic_bytes": nbytes,
                           "hbm_frac": nbytes / (nms / 1e3) / 1e9 / peak_gbs}
    except Exception as exc:
        line["nearest"] = {"error": repr(exc)}

    # ------------------------------------------------------- e2e (host buffers)
    if not args.no_e2e:
        hq = torch.from_numpy(qs).pin_memory()
        h_counts = torch.empty(args.queries, dtype=torch.int32).pin_memory()
        h_offsets = torch.empty(args.queries, dtype=torch.int64).pin_memory()
        h_idx = torch.empty(K + 16, dtype=torch.int32).pin_memory()
        h_dist = torch.empty(K + 16, dtype=torch.float64).pin_memory()
        res2 = RangeResult(ctx)
        from rrtqx_3d_b200 import _abi as A

        def e2e_step():
            # the call a user of the C ABI makes: host queries in, host lists out
            _, tot = tree.range_query(hq.numpy(), r, want_dist=True, result=res2)
            A.check(ctx.L.rrtqx_range_result_layout(res2.h, h_counts.data_ptr(), h_offsets.data_ptr()), ctx.h)
            A.check(ctx.L.rrtqx_range_result_fetch(res2.h, h_idx.data_ptr(), h_dist.data_ptr()), ctx.h)
            return tot

        e2e_step()
        n_e2e = max(2, min(args.steps, 3))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record(stream)
        for _ in range(n_e2e):
            tot = e2e_step()
        eb.record(stream)
        torch.cuda.synchronize()
        e2e_ms = ea.elapsed_time(eb) / n_e2e
        e2e_wall_ms = 1e3 * (time.perf_counter() - t0) / n_e2e
        if world > 1:
            tmax = torch.tensor([e2e_ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            e2e_ms = float(tmax.item())
        line["e2e"] = {"value": world * args.queries / (e2e_ms / 1e3), "unit": "queries/s",
                       "h2d_bytes_per_step": args.queries * 24,
                       "d2h_bytes_per_step": args.queries * 12 + tot * 12,
                       "ms_per_step": e2e_ms, "wall_ms_per_step": e2e_wall_ms,
                       "note": "pinned host queries -> rrtqx_range_query_batch -> counts/offsets/idx/dist copied to pinned host (rrtqx_host_alloc gives a Julia caller the same kind of memory)"}
        del h_idx, h_dist
        if world == 1:
            # the same call with ORDINARY (pageable) host arrays -- what a Julia caller passes when it hands over plain
            # `Vector`s instead of memory from rrtqx_host_alloc; the driver stages every copy
            try:
                pq = np.array(qs, copy=True)
                p_counts, p_offsets = np.empty(args.queries, np.int32), np.empty(args.queries, np.int64)
                p_idx, p_dist = np.empty(K + 16, np.int32), np.empty(K + 16, np.float64)

                def pageable_step():
                    _, tot = tree.range_query(pq, r, want_dist=True, result=res2)
                    A.check(ctx.L.rrtqx_range_result_layout(res2.h, p_counts.ctypes.data, p_offsets.ctypes.data), ctx.h)
                    A.check(ctx.L.rrtqx_range_result_fetch(res2.h, p_idx.ctypes.data, p_dist.ctypes.data), ctx.h)
                    return tot

                pageable_step()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(2):
                    pageable_step()
                torch.cuda.synchronize()
                pms = 1e3 * (time.perf_counter() - t0) / 2
                line["e2e_pageable"] = {"value": args.queries / (pms / 1e3), "unit": "queries/s", "ms_per_step": pms,
                                        "note": "as e2e, but every host array is ordinary pageable memory (wall clock, 2 steps)"}
                del p_idx, p_dist
            except Exception as exc:
                line["e2e_pageable"] = {"error": repr(exc)}
        res2.close()

    # ------------------------------------------------- extra: C3 obstacle-add sweep
    if not args.no_sweep and rank == 0:
        try:
            src, dst, parent = build_c3_edges(tree, pts, args.sweep_edge_radius)
            E = EdgeSet(tree)
            E.upload(src, dst, parent)
            centers, radii = W.c3_obstacles(args.sweep_obstacles)
            S = SphereSet(ctx, centers, radii)
            ids = np.arange(args.sweep_obstacles, dtype=np.int32)
            sres = SweepResult(ctx)
            from rrtqx_3d_b200 import _abi as A
            times, times_stats = [], []
            for it in range(3 + args.steps):
                flush.zero_()
                E.add_sweep(S, ids, W.ROBOT_RADIUS, W.DELTA, flags=A.SWEEP_STATS, result=sres)   # node-centric + statistics
                if it >= 3:
                    times_stats.append(ctx.last_phase_ms("add_sweep"))
            n_eh, n_nh, n_cand, n_tests = sres.sizes()
            for it in range(3 + args.steps):
                flush.zero_()
                E.add_sweep(S, ids, W.ROBOT_RADIUS, W.DELTA, result=sres)                        # edge-centric (default)
                if it >= 3:
                    times.append(ctx.last_phase_ms("add_sweep"))
            assert sres.sizes()[:2] == (n_eh, n_nh)
            sms = float(np.mean(times))
            # the planner's real call: ONE new obstacle (addNewObstacle, DRRT_Q.jl:3220) against the same resident graph
            one_ms, one_hits = [], 0
            for k in range(16):
                E.add_sweep(S, ids[k:k + 1], W.ROBOT_RADIUS, W.DELTA, result=sres)
                one_ms.append(ctx.last_phase_ms("add_sweep"))
                one_hits += sres.sizes()[0]
            n_e = len(src)
            sbytes = args.nodes * 24 + n_e * 8 + args.sweep_obstacles * 40 + n_e * 1 + (n_eh + n_nh) * 4
            # C5-style batch: explicitEdgeCheck(S, edge) of every edge against all 256 active spheres
            dsrc, ddst = torch.from_numpy(src).cuda(), torch.from_numpy(dst).cuda()
            dflag = torch.empty(len(src), dtype=torch.uint8, device="cuda")
            from rrtqx_3d_b200.device import edge_check_batch
            et = []
            for it in range(3 + args.steps):
                flush.zero_()
                edge_check_batch(tree, S, dsrc, ddst, W.ROBOT_RADIUS, n_edges=len(src), out=dflag)
                if it >= 3:
                    et.append(ctx.last_phase_ms("edge_check"))
            ems = float(np.mean(et))
            # the same check over the RESIDENT edge set (rrtqx_edges_check_batch: per-edge records prepared at upload)
            rflag = torch.empty(len(src), dtype=torch.uint8, device="cuda")
            rt = []
            for it in range(3 + args.steps):
                flush.zero_()
                E.check_all(S, W.ROBOT_RADIUS, out=rflag.data_ptr())
                if it >= 3:
                    rt.append(ctx.last_phase_ms("edges_check"))
            rms = float(np.mean(rt))
            resident_equal = bool(torch.equal(rflag, dflag))
            # CPU side of the same batch: the oracle's explicitEdgeCheck loop (front-to-back over the obstacle list,
            # early exit) on a bounded sample of the edges, all host threads
            cpu_edge = None
            if not args.no_cpu:
                import oracle
                nthr = os.cpu_count() or 1
                sph, ns = oracle.make_spheres(centers, radii)
                hp = np.ascontiguousarray(pts)

                def _cpu_edges(n):
                    o = np.zeros(n, dtype=np.uint8)
                    t0 = time.perf_counter()
                    oracle.lib().orc_edge_check_batch(sph, ns, oracle._p(hp, oracle.c_f64p), 3, oracle._p(src, oracle.c_i32p),
                                                      oracle._p(dst, oracle.c_i32p), 0, n, W.ROBOT_RADIUS, 0,
                                                      oracle._p(o, oracle.c_u8p), nthr)
                    return time.perf_counter() - t0, o
                dt, _ = _cpu_edges(min(len(src), 20000 * nthr))
                n_s = int(min(len(src), max(20000 * nthr, min(len(src), 20000 * nthr) / dt * 4.0)))
                dt, flags_cpu = _cpu_edges(n_s)
                cpu_edge = {"value": n_s / dt, "unit": "edges/s", "cores": nthr, "kind": "port",
                            "sample": f"first {n_s} of {len(src)} C3 edges vs 256 spheres, {dt:.1f}s timed",
                            "matches_gpu": bool(np.array_equal(flags_cpu, dflag[:n_s].cpu().numpy()))}
            line["edge_batch"] = {"cpu_baseline": cpu_edge,
                                  "workload": "explicitEdgeCheck(S, edge) for every C3 edge against all 256 spheres (device-resident)",
                                  "edges": len(src), "obstacles": args.sweep_obstacles, "ms": ems,
                                  "resident_ms": rms, "resident_edges_per_s": len(src) / (rms / 1e3),
                                  "resident_equals_batch": resident_equal,
                                  "resident_algorithmic_bytes": len(src) * 17,
                                  "resident_hbm_frac": len(src) * 17 / (rms / 1e3) / 1e9 / peak_gbs,
                                  "edges_per_s": len(src) / (ems / 1e3),
                                  "edge_obstacle_pairs_per_s": len(src) * args.sweep_obstacles / (ems / 1e3),
                                  "colliding_edges": int(dflag.sum().item()),
                                  "algorithmic_bytes": len(src) * 9 + args.nodes * 32,
                                  "hbm_frac": (len(src) * 9 + args.nodes * 32) / (ems / 1e3) / 1e9 / peak_gbs}
            # FP64 side of the bound (SURVEY 8d: report max(B/BW, F/FP64)).  The reference evaluates `pair_checks`
            # (edge, obstacle) pairs (those that pass its start-node filter), 27 separately rounded FP64 operations
            # each (3 sub, 3 mul + 3 add dot, 1 div, 3 mul + 3 add closest point, 3 sub + 3 mul + 2 add radicand) +
            # 12 for a conservative FP64 reject = 39; the statistics kernel executes exactly that, and its fraction of
            # the unfused FP64 rate (half the measured FMA flop rate) is reported.  The default two-stage path culls
            # in FP32 on cover lists and runs the exact test only on the surviving pairs, so for it the reference-
            # equivalent pair rate is the meaningful figure, not an FP64 utilisation.
            fp64_tflops = ctx.measure_fp64_peak()
            ops = n_tests * 39.0
            line["fp64_peak_tflops_measured"] = fp64_tflops
            line["edge_sweep"] = {"workload": "C3 obstacle-add sweep: 256 spheres vs all out-edges + parent edges of the 1M-node tree",
                                  "fp64_ops_statistics_kernel": ops,
                                  "fp64_frac_of_unfused_peak_statistics_kernel": ops / (float(np.mean(times_stats)) / 1e3) / (fp64_tflops / 2 * 1e12),
                                  "edges": n_e, "obstacles": args.sweep_obstacles, "pair_checks": n_tests,
                                  "candidate_nodes": n_cand, "blocked_edges": n_eh, "orphans": n_nh, "ms": sms,
                                  "single_obstacle_ms": float(np.median(one_ms)), "single_obstacle_mean_blocked_edges": one_hits / 16,
                                  "ms_with_statistics_kernel": float(np.mean(times_stats)),
                                  "edges_per_s": n_e / (sms / 1e3), "pair_checks_per_s": n_tests / (sms / 1e3),
                                  "algorithmic_bytes": sbytes, "hbm_frac": sbytes / (sms / 1e3) / 1e9 / peak_gbs}
        except Exception as exc:  # the headline line must still be printed
            line["edge_sweep"] = {"error": repr(exc)}

    # ------------------------------------------------- C5: sharded edge-check batch + independent instances
    if not args.no_c5:
        try:
            from rrtqx_3d_b200.device import edge_check_batch
            from rrtqx_3d_b200.sharding import shard_bounds
            src, dst, _ = build_c3_edges(tree, pts, args.sweep_edge_radius)     # every rank: same edge set
            centers, radii = W.c3_obstacles(args.sweep_obstacles)
            S5 = SphereSet(ctx, centers, radii)
            c5comm = comm if comm is not None else Comm.local([ctx])
            words, _ = c5comm.packed_words(len(src))
            dsrc, ddst = torch.from_numpy(src).cuda(), torch.from_numpy(dst).cuda()   # replicated edge list
            packed = torch.zeros(words, dtype=torch.int32, device="cuda")             # ALL flags, bit-packed, on every rank
            torch.cuda.synchronize()
            evs = []
            for it in range(3 + args.steps):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                # rank g checks word shard g; the packed words are gathered inside the library (NCCL, in place)
                c5comm.edge_check_sharded([tree], [S5], [dsrc], [ddst], len(src), W.ROBOT_RADIUS, [packed])
                b.record(stream)
                b.synchronize()
                if it >= 3:
                    evs.append(a.elapsed_time(b))
            ems = float(np.mean(evs))
            # weak-scaled form of the same check: EVERY rank holds the 9.85M-edge graph resident and checks all of it
            # (world x 9.85M edges per step, rrtqx_edges_check_batch); the fixed-size result that is exchanged is each
            # rank's count of colliding edges
            E5 = EdgeSet(tree)
            E5.upload(src, dst, None)
            wflag = torch.empty(len(src), dtype=torch.uint8, device="cuda")
            wevs = []
            for it in range(3 + args.steps):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                E5.check_all(S5, W.ROBOT_RADIUS, out=wflag.data_ptr())
                b.record(stream)
                b.synchronize()
                if it >= 3:
                    wevs.append(a.elapsed_time(b))
            wms = float(np.mean(wevs))
            wcount = int(wflag.sum().item())
            E5.close()
            done, secs = c5_instances(ctx, rank, world, args.c5_instances, args.c5_iterations)
            if world > 1:
                tt = torch.tensor([ems, secs, wms], device="cuda", dtype=torch.float64)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                ems, secs, wms = float(tt[0].item()), float(tt[1].item()), float(tt[2].item())
                dd = torch.tensor([done], device="cuda", dtype=torch.int64)
                dist.all_reduce(dd)
                done = int(dd.item())
            pk = packed.cpu().numpy().view(np.uint32)
            colliding = int(np.unpackbits(pk.view(np.uint8))[:].sum())   # padding words are zero
            c5_info = c5comm.info()
            if comm is None:
                c5comm.close()
            line["c5"] = {"workload": "C5: C3 edge set sharded contiguously over the ranks (tree + 256 spheres replicated, "
                                      "bit-packed flags gathered inside the library: rrtqx_edge_check_batch_sharded) and "
                                      "independent C1-style planning instances round-robin",
                          "comm": c5_info,
                          "edges": len(src), "edge_shards": world, "edge_batch_ms": ems,
                          "edge_weak_ms": wms, "edge_weak_edges_per_s": world * len(src) / (wms / 1e3),
                          "edge_weak_colliding_edges_rank0": wcount,
                          "edge_weak_note": "every rank checks its own resident copy of the graph (world x edges per step)",
                          "edges_per_s": len(src) / (ems / 1e3), "colliding_edges": colliding, "scaling": "strong",
                          "instances": args.c5_instances, "iterations_per_instance": args.c5_iterations,
                          "instance_seconds": secs, "planner_iterations_per_s": done / secs}
        except Exception as exc:
            line["c5"] = {"error": repr(exc)}

    if not args.no_c4 and rank == 0 and world == 1:
        try:
            line["dubins"] = c4_dubins(ctx, args.c4_edges, max(3, min(args.steps, 10)))
        except Exception as exc:
            line["dubins"] = {"error": repr(exc)}

    if not args.no_c1 and rank == 0 and world == 1:
        try:
            line["planner_iteration"] = c1_replay(ctx, args.c1_iterations)
        except Exception as exc:
            line["planner_iteration"] = {"error": repr(exc)}

    # ---------------------------------------------------------- CPU baseline
    if not args.no_cpu and rank == 0 and world == 1:
        base, otree = cpu_range_baseline(pts, qs, r)
        line["cpu_baseline"] = base
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
