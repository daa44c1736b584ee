"""Lock-step Dubins planner iterations for many independent trees against the serial loop.

N city-block instances (config C4's [x y t theta] tree with the heading wrapped at 2 pi, seeds 1..N) grow from one
pose among workloads.c4_city_blocks with r = 1.06, delta = 1 and RRTQX_EXTEND_SATURATE; the saturated point is
inserted iff some forward edge is free and has a finite length.  Two forms run in the same process, alternating:
  (a) serial:    for every instance, for every iteration: extend_query_dubins + insert;
  (b) lock-step: for every iteration, one extend_query_dubins_multi over all instances + one insert_multi of the
                 accepted points.
Each instance sees the same sequence of calls either way.  For every N one JSON line: iterations/s of both forms
(time inside the library calls and their argument glue; hashing is outside the timed spans), the median round time
of (b), and a hash per form of every iteration's outputs (nearest, point, ball, per-edge dist / type / collision and
trajectory rows).  Exits non-zero if the hashes differ.  Needs a B200: there is no fallback.

    python scripts/exp_lockstep_dubins.py [--sizes 1,4,16,64,148,296] [--iterations 500] [--reps 2] [--out f]
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rrtqx_3d_b200 import _abi as A  # noqa: E402
from rrtqx_3d_b200 import workloads as W  # noqa: E402
from rrtqx_3d_b200.device import Context, DeviceTree, DubinsResult, PolygonSet  # noqa: E402

TWO_PI = 2.0 * math.pi
ROOT = np.array([0.0, 0.0, 0.0, 1.0])     # a pose in a street of the city-block world
R, DELTA, RHO, R_TURN = 1.06, 1.0, 0.5, 1.0
CAPACITY = 1024
FLAGS = A.EXTEND_SATURATE


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power = [x.strip() for x in out.split(",")]
    return name, power


def samples_for(seed, n):
    return W.uniform_points(seed, n, [-50.0, -50.0, 0.0, 0.0], [50.0, 50.0, 0.0, TWO_PI])


class Digest:
    """Per-instance hash of every iteration's outputs; neighbour lists are sets, so they are hashed in node order
    with each neighbour's two edges and their rows."""

    def __init__(self, n):
        self.h = [hashlib.blake2b(digest_size=16) for _ in range(n)]

    def add(self, i, ni, nd, point, cnt, idx, dist, edist, etype, ecol, ptr, xy):
        h = self.h[i]
        h.update(np.array([ni, cnt], dtype=np.int64).tobytes())
        h.update(np.array([nd], dtype=np.float64).tobytes())
        h.update(np.ascontiguousarray(point, dtype=np.float64).tobytes())
        for k in np.argsort(idx, kind="stable"):
            h.update(np.array([idx[k]], dtype=np.int64).tobytes())
            h.update(np.array([dist[k]], dtype=np.float64).tobytes())
            for e in (2 * k, 2 * k + 1):
                h.update(np.array([edist[e]], dtype=np.float64).tobytes())
                h.update(np.array([etype[e], ecol[e]], dtype=np.int64).tobytes())
                h.update(np.ascontiguousarray(xy[ptr[e]:ptr[e + 1]]).tobytes())

    def hexdigest(self):
        t = hashlib.blake2b(digest_size=16)
        for h in self.h:
            t.update(h.digest())
        return t.hexdigest()


def new_tree(ctx):
    t = DeviceTree(ctx, 4, wraps=(3,), wrap_points=(TWO_PI,))
    t.insert(ROOT)
    return t


def run_serial(ctx, P, samples, n_iter):
    n = len(samples)
    dig = Digest(n)
    L = ctx.L
    ptr = A.ptr
    idx, dist = np.empty(CAPACITY, np.int32), np.empty(CAPACITY)
    edist, etype, ecol = np.empty(2 * CAPACITY), np.empty(2 * CAPACITY, np.int32), np.empty(2 * CAPACITY, np.uint8)
    ni, nd, cnt = A.i32(0), A.f64(0.0), A.i32(0)
    traj = DubinsResult(ctx)
    secs = 0.0
    for i in range(n):
        t = new_tree(ctx)
        ctx.sync()
        for it in range(n_iter):
            p = np.array(samples[i][it], copy=True)
            t0 = time.perf_counter()
            A.check(L.rrtqx_extend_query_dubins(t.h, P.h, ptr(p), DELTA, R, RHO, R_TURN, FLAGS, CAPACITY,
                                                C.byref(ni), C.byref(nd), C.byref(cnt), ptr(idx), ptr(dist),
                                                ptr(edist), ptr(etype), ptr(ecol), C.byref(traj.h)), ctx.h)
            m = min(int(cnt.value), CAPACITY)
            accept = bool(((ecol[0:2 * m:2] == 0) & np.isfinite(edist[0:2 * m:2])).any())
            if accept:
                t.insert(p)
            secs += time.perf_counter() - t0
            _, _, tp, xy = traj.fetch()
            dig.add(i, int(ni.value), float(nd.value), p, int(cnt.value), idx[:m], dist[:m], edist[:2 * m],
                    etype[:2 * m], ecol[:2 * m], tp, xy)
        t.close()
    return secs, None, dig.hexdigest()


def run_lockstep(ctx, P, samples, n_iter):
    n = len(samples)
    dig = Digest(n)
    L = ctx.L
    ptr = A.ptr
    trees = [new_tree(ctx) for _ in range(n)]
    handles = np.array([t.h.value for t in trees], dtype=np.uint64)
    poly_handles = np.full(n, P.h.value, dtype=np.uint64)
    ctx.sync()
    ni, nd, cnt = np.empty(n, np.int32), np.empty(n), np.empty(n, np.int32)
    idx, dist = np.empty(n * CAPACITY, np.int32), np.empty(n * CAPACITY)
    edist, etype = np.empty(2 * n * CAPACITY), np.empty(2 * n * CAPACITY, np.int32)
    ecol = np.empty(2 * n * CAPACITY, np.uint8)
    ranges = np.full(n, R)
    index_out = np.empty(n, np.int32)
    pts_all = np.ascontiguousarray(np.stack(samples, axis=1))   # n_iter x n x 4
    traj = DubinsResult(ctx)
    rounds = []
    for it in range(n_iter):
        pts = np.array(pts_all[it], copy=True)
        t0 = time.perf_counter()
        A.check(L.rrtqx_extend_query_dubins_multi(ptr(handles), ptr(poly_handles), n, ptr(pts), ptr(ranges), DELTA,
                                                  RHO, R_TURN, FLAGS, CAPACITY, ptr(ni), ptr(nd), ptr(cnt), ptr(idx),
                                                  ptr(dist), ptr(edist), ptr(etype), ptr(ecol), C.byref(traj.h)),
                ctx.h)
        m = np.minimum(cnt, CAPACITY)
        acc = np.zeros(n, dtype=bool)
        for i in range(n):
            e = 2 * i * CAPACITY
            acc[i] = ((ecol[e:e + 2 * m[i]:2] == 0) & np.isfinite(edist[e:e + 2 * m[i]:2])).any()
        k = int(np.count_nonzero(acc))
        if k:
            # the arrays must outlive the call: ptr() of a temporary would hand freed memory to the library
            sub, sub_pts = (handles, pts) if k == n else (handles[acc], np.ascontiguousarray(pts[acc]))
            A.check(L.rrtqx_tree_insert_multi(ptr(sub), k, ptr(sub_pts), ptr(index_out)), ctx.h)
        rounds.append(time.perf_counter() - t0)
        _, _, tp, xy = traj.fetch()
        first = 0
        for i in range(n):
            a, e = i * CAPACITY, 2 * i * CAPACITY
            dig.add(i, int(ni[i]), float(nd[i]), pts[i], int(cnt[i]), idx[a:a + m[i]], dist[a:a + m[i]],
                    edist[e:e + 2 * m[i]], etype[e:e + 2 * m[i]], ecol[e:e + 2 * m[i]],
                    tp[first:first + 2 * m[i] + 1] - tp[first], xy[tp[first]:])
            first += 2 * int(m[i])
    for t in trees:
        t.close()
    return float(np.sum(rounds)), float(np.median(rounds)), dig.hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,4,16,64,148,296")
    ap.add_argument("--iterations", type=int, default=500)
    ap.add_argument("--reps", type=int, default=2, help="alternating (a, b) passes per size; the best time is kept")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    ctx = Context(0)                    # raises without a usable B200: no fallback
    name, power = gpu_info()
    P = PolygonSet(ctx)
    P.upload(W.c4_city_blocks())
    ok = True
    for n in [int(x) for x in args.sizes.split(",")]:
        samples = [samples_for(1 + i, args.iterations) for i in range(n)]
        run_lockstep(ctx, P, [s[:20] for s in samples], 20)   # warm-up of both forms' modules and buffers at this size
        run_serial(ctx, P, samples[:1], 20)
        best_a, best_b, med_b, ha, hb = np.inf, np.inf, None, set(), set()
        for _ in range(args.reps):
            sa, _, h = run_serial(ctx, P, samples, args.iterations)
            best_a = min(best_a, sa)
            ha.add(h)
            sb, mb, h = run_lockstep(ctx, P, samples, args.iterations)
            if sb < best_b:
                best_b, med_b = sb, mb
            hb.add(h)
        iters = n * args.iterations
        same = len(ha) == 1 and ha == hb
        ok &= same
        line = {"experiment": "lockstep_dubins", "gpu": name, "power_limit": power, "instances": n,
                "iterations_per_instance": args.iterations, "reps": args.reps,
                "serial_iter_per_s": iters / best_a, "lockstep_iter_per_s": iters / best_b,
                "speedup": best_a / best_b, "lockstep_median_round_us": med_b * 1e6,
                "hash_serial": sorted(ha), "hash_lockstep": sorted(hb), "hashes_equal": same}
        print(json.dumps(line), flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(json.dumps(line) + "\n")
    if not ok:
        print("output hashes differ between the serial and the lock-step form", file=sys.stderr)
        sys.exit(1)


if __name__ == "__main__":
    main()
