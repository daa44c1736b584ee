"""Config C4 planner iteration: the fused rrtqx_extend_query_dubins against the same work composed from the batch
entry points (nearest -> Dubins saturate -> range query -> Dubins trajectories -> Dubins edge check) and against the
oracle on one CPU thread (every 25th iteration).  Prints one JSON line with the card's name and power limit.

  (a) c4:    a 2e5-pose C4 tree ([-50,50]^2 x {0} x [0,2pi), theta wrapped), r = 1.06, city blocks; 2000 replayed
             samples, each saturated (delta 1.0) and inserted through rrtqx_tree_insert.
  (b) paper: delta = 10, gamma = 100 (r = min(gamma (log n / n)^(1/4), delta) = 10 > pi), a tree grown from one pose
             by 3000 iterations among a reference polygon file plus balls.

Both paths run on every iteration, alternating which goes first, and their outputs are compared; the script exits
non-zero if they differ.  Times are host wall clock per call (each call ends with its results on the host).
Usage: python scripts/exp_c4_iteration.py [--iters-a 2000] [--iters-b 3000] [--out FILE]"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from rrtqx_3d_b200 import _abi as A  # noqa: E402
from rrtqx_3d_b200 import workloads as W  # noqa: E402
from rrtqx_3d_b200.device import (Context, DeviceTree, DubinsResult, PolygonSet, RangeResult,  # noqa: E402
                                  extend_query_dubins, extend_query_dubins_composed)
from rrtqx_3d_b200.formats import read_polygon_obstacles  # noqa: E402

TWO_PI = 2.0 * math.pi
RHO, R_TURN = 0.5, 1.0


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return name, power


def same(a, b):
    """Fused and composed outputs agree bit for bit (neighbour lists compared as sets, edges per neighbour)."""
    bits = lambda x: np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)
    if (a.nearest_idx, a.count) != (b.nearest_idx, b.count) or bits([a.nearest_dist])[0] != bits([b.nearest_dist])[0]:
        return False
    if not np.array_equal(bits(a.point), bits(b.point)):
        return False
    ga, gb = np.argsort(a.idx, kind="stable"), np.argsort(b.idx, kind="stable")
    ea = np.stack([2 * ga, 2 * ga + 1], axis=1).reshape(-1)
    eb = np.stack([2 * gb, 2 * gb + 1], axis=1).reshape(-1)
    return (np.array_equal(a.idx[ga], b.idx[gb]) and np.array_equal(bits(a.dist[ga]), bits(b.dist[gb]))
            and np.array_equal(bits(a.edge_dist[ea]), bits(b.edge_dist[eb]))
            and np.array_equal(a.edge_type[ea], b.edge_type[eb])
            and np.array_equal(a.edge_collide[ea], b.edge_collide[eb]))


def oracle_iteration(orc, orc_obs, pts, q, r, delta):
    """The same iteration on one CPU thread: kdFindNearest, saturate, kdFindWithinRange, calculateTrajectory and
    the Dubins edge check of both edges per neighbour, OR-ed over the obstacles."""
    import ctypes as C
    L = oracle.lib()
    f = lambda a: oracle._p(np.ascontiguousarray(a, dtype=np.float64), oracle.c_f64p)
    ni, _ = orc.find_nearest(q)
    p = oracle.saturate_dubins(q, pts[ni], delta)
    idx, _ = orc.find_within_range(r, p)
    orc.empty(idx)
    for i in idx:
        for s, g in ((p, pts[i]), (pts[i], p)):
            _, _, tr = oracle.dubins_trajectory(s, g, R_TURN)
            for ob in orc_obs:
                if L.orc_edge_check_dubins(C.byref(ob), f(s[:2]), f(g[:2]), f(tr), len(tr), RHO, R_TURN):
                    break


def run(ctx, regime, n_iter):
    from test_gpu_collision import _orc_obstacles_2d
    P = PolygonSet(ctx)
    if regime == "c4":
        P.upload(W.c4_city_blocks())
        base = W.uniform_points(4, 200_000, [-50.0, -50.0, 0.0, 0.0], [50.0, 50.0, 0.0, TWO_PI])
        delta = 1.0
    else:
        obs = read_polygon_obstacles(os.path.join(ROOT, "tests", "golden", "ref_rand_Static.txt"))
        P.upload([("polygon", o["polygon"]) for o in obs] + [("ball", (5.0, 5.0), 3.0), ("ball", (-20.0, 31.0), 4.0),
                                                        ("ball", (30.0, -12.0), 2.5)])
        base = np.array([[10.0, 0.0, 0.0, 1.0]])   # in free space: the origin lies inside a polygon of this file
        delta = 10.0
    orc_obs = _orc_obstacles_2d(P)
    t = DeviceTree(ctx, 4, wraps=(3,), wrap_points=(TWO_PI,))
    t.insert_batch(base)
    orc = oracle.KDTree(4, wraps=[3], wrap_points=[TWO_PI])
    orc.insert_batch(base)
    pts = np.zeros((len(base) + n_iter, 4))
    pts[:len(base)] = base
    n = len(base)
    samples = W.uniform_points(77 if regime == "c4" else 78, n_iter, [-50.0, -50.0, 0.0, 0.0],
                               [50.0, 50.0, 0.0, TWO_PI])
    fr, cr, rr = DubinsResult(ctx), DubinsResult(ctx), RangeResult(ctx)
    flags = A.EXTEND_SATURATE
    t_f, t_c, t_o, ks, mismatches = [], [], [], [], 0
    for it in range(n_iter):
        r = 1.06 if regime == "c4" else (min(100.0 * (math.log(n) / n) ** 0.25, delta) if n > 1 else delta)
        q = samples[it]
        order = (0, 1) if it % 2 == 0 else (1, 0)
        out = [None, None]
        for which in order:
            t0 = time.perf_counter()
            if which == 0:
                out[0] = extend_query_dubins(t, P, q, r, RHO, R_TURN, delta=delta, flags=flags, trajectories=fr)
            else:
                out[1] = extend_query_dubins_composed(t, P, q, r, RHO, R_TURN, pts[:n], delta=delta, flags=flags,
                                                      trajectories=cr, range_result=rr)
            (t_f if which == 0 else t_c).append(time.perf_counter() - t0)
        a, b = out
        if not same(a, b):
            mismatches += 1
        if it % 25 == 0:
            t0 = time.perf_counter()
            oracle_iteration(orc, orc_obs, pts[:n], q, r, delta)
            t_o.append(time.perf_counter() - t0)
        ks.append(a.count)
        if regime == "c4" or ((a.edge_collide[0::2] == 0) & np.isfinite(a.edge_dist[0::2])).any():
            t.insert(a.point)
            orc.insert(a.point)
            pts[n] = a.point
            n += 1
    w = lambda v: v[len(v) // 10:] if len(v) > 20 else v   # the first tenth warms up modules and buffers
    us = lambda v: round(1e6 * float(np.median(w(v))), 1)
    return {"regime": regime, "iterations": n_iter, "final_tree": n, "r_last": r, "mean_k": round(float(np.mean(ks)), 1),
            "fused_us_median": us(t_f), "fused_us_mean": round(1e6 * float(np.mean(w(t_f))), 1),
            "composed_us_median": us(t_c), "composed_us_mean": round(1e6 * float(np.mean(w(t_c))), 1),
            "oracle_1thread_us_median": us(t_o), "oracle_samples": len(t_o),
            "speedup_vs_composed": round(float(np.median(w(t_c)) / np.median(w(t_f))), 2),
            "mismatches": mismatches}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters-a", type=int, default=2000)
    ap.add_argument("--iters-b", type=int, default=3000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    name, power = card()
    ctx = Context(0)
    res = [run(ctx, "c4", args.iters_a), run(ctx, "paper", args.iters_b)]
    line = json.dumps({"experiment": "c4_iteration", "device": name, "power_limit": power, "results": res})
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    if any(r["mismatches"] for r in res):
        sys.exit("fused and composed outputs differ")


if __name__ == "__main__":
    main()
