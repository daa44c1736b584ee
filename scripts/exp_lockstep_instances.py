"""Lock-step planner iterations for many independent trees against today's serial loop.

C5a-style instances (seeds 1..N, building2 spheres, the shrinking ball, insert iff the point check passes, as
bench.py's c5_instances) run two ways in the same process, alternating:
  (a) serial:    for every instance, for every iteration: extend_query + insert (one launch + one wait each);
  (b) lock-step: for every iteration, one extend_query_multi over all instances + one insert_multi of the
                 accepted samples (one launch + one wait per round for the query, one launch for the inserts).
Each instance sees the same sequence of calls either way.  For every N one JSON line: iterations/s of both forms
(time inside the library calls and their argument glue; hashing is outside the timed spans), the median round time
of (b), and a hash of every iteration's outputs per form.  Exits non-zero if the hashes differ.  Needs a B200: there
is no fallback.

    python scripts/exp_lockstep_instances.py [--sizes 1,4,16,64,148,296] [--iterations 1000] [--reps 2] [--out f]
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rrtqx_3d_b200 import _abi as A  # noqa: E402
from rrtqx_3d_b200 import workloads as W  # noqa: E402
from rrtqx_3d_b200.device import Context, DeviceTree, SphereSet, extend_query  # noqa: E402

ROOT_NODE = np.array([4.0, 16.5, -7.5])   # bench.py c5_instances
CAPACITY = 8192
FLAGS = A.CHECK_QUICK_PASS


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power = [x.strip() for x in out.split(",")]
    return name, power


class Digest:
    """Per-instance hash of every iteration's outputs; neighbour lists are sets, so they are hashed in node order."""

    def __init__(self, n):
        self.h = [hashlib.blake2b(digest_size=16) for _ in range(n)]

    def add(self, i, ni, nd, pc, ce, cnt, idx, dist, fwd, rev):
        o = np.argsort(idx, kind="stable")
        h = self.h[i]
        h.update(np.array([ni, cnt, int(pc)], dtype=np.int64).tobytes())
        h.update(np.array([nd, ce], dtype=np.float64).tobytes())
        h.update(np.ascontiguousarray(idx[o]).tobytes())
        h.update(np.ascontiguousarray(dist[o]).tobytes())
        h.update(np.ascontiguousarray(fwd[o]).tobytes())
        h.update(np.ascontiguousarray(rev[o]).tobytes())

    def hexdigest(self):
        t = hashlib.blake2b(digest_size=16)
        for h in self.h:
            t.update(h.digest())
        return t.hexdigest()


def run_serial(ctx, S, samples, n_iter):
    n = len(samples)
    dig = Digest(n)
    bufs = (np.empty(CAPACITY, np.int32), np.empty(CAPACITY, np.float64), np.empty(CAPACITY, np.uint8),
            np.empty(CAPACITY, np.uint8))
    secs = 0.0
    for i in range(n):
        t = DeviceTree(ctx, 3)
        t.insert(ROOT_NODE)
        ctx.sync()
        size = 1
        for it in range(n_iter):
            p = samples[i][it]
            r = W.shrinking_ball_radius(size, 3, W.DELTA, W.BALL_CONSTANT)
            t0 = time.perf_counter()
            res = extend_query(t, S, p, r, W.ROBOT_RADIUS, FLAGS, capacity=CAPACITY, bufs=bufs)
            if not res.point_collides:
                t.insert(p)
            secs += time.perf_counter() - t0
            if not res.point_collides:
                size += 1
            dig.add(i, res.nearest_idx, res.nearest_dist, res.point_collides, res.point_cert, res.count, res.idx,
                    res.dist, res.fwd, res.rev)
        t.close()
    return secs, None, dig.hexdigest()


def run_lockstep(ctx, S, samples, n_iter):
    n = len(samples)
    dig = Digest(n)
    L = ctx.L
    trees = [DeviceTree(ctx, 3) for _ in range(n)]
    handles = np.array([t.h.value for t in trees], dtype=np.uint64)
    sphere_handles = np.full(n, S.h.value, dtype=np.uint64)
    for t in trees:
        t.insert(ROOT_NODE)
    ctx.sync()
    sizes = np.ones(n, dtype=np.int64)
    ni, nd = np.empty(n, np.int32), np.empty(n, np.float64)
    pc, ce, cnt = np.empty(n, np.uint8), np.empty(n, np.float64), np.empty(n, np.int32)
    idx, dist = np.empty(n * CAPACITY, np.int32), np.empty(n * CAPACITY, np.float64)
    fwd, rev = np.empty(n * CAPACITY, np.uint8), np.empty(n * CAPACITY, np.uint8)
    index_out = np.empty(n, np.int32)
    pts_all = np.ascontiguousarray(np.stack(samples, axis=1))   # n_iter x n x 3
    rounds = []
    ptr = A.ptr
    for it in range(n_iter):
        pts = pts_all[it]
        ranges = np.array([W.shrinking_ball_radius(int(s), 3, W.DELTA, W.BALL_CONSTANT) for s in sizes])
        t0 = time.perf_counter()
        A.check(L.rrtqx_extend_query_multi(ptr(handles), ptr(sphere_handles), n, ptr(pts), ptr(ranges),
                                           W.ROBOT_RADIUS, FLAGS, CAPACITY, ptr(ni), ptr(nd), ptr(pc), ptr(ce),
                                           ptr(cnt), ptr(idx), ptr(dist), ptr(fwd), ptr(rev)), ctx.h)
        acc = pc == 0
        k = int(np.count_nonzero(acc))
        if k:
            # the arrays must outlive the call: ptr() of a temporary would hand freed memory to the library
            sub, sub_pts = (handles, pts) if k == n else (handles[acc], pts[acc])
            A.check(L.rrtqx_tree_insert_multi(ptr(sub), k, ptr(sub_pts), ptr(index_out)), ctx.h)
        rounds.append(time.perf_counter() - t0)
        sizes += acc
        for i in range(n):
            a = i * CAPACITY
            b = a + min(int(cnt[i]), CAPACITY)
            dig.add(i, int(ni[i]), float(nd[i]), bool(pc[i]), float(ce[i]), int(cnt[i]), idx[a:b], dist[a:b],
                    fwd[a:b], rev[a:b])
    for t in trees:
        t.close()
    return float(np.sum(rounds)), float(np.median(rounds)), dig.hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,4,16,64,148,296")
    ap.add_argument("--iterations", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=2, help="alternating (a, b) passes per size; the best time is kept")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    ctx = Context(0)                    # raises without a usable B200: no fallback
    name, power = gpu_info()
    centers, radii, _ = W.building2_spheres()
    S = SphereSet(ctx, centers, radii)
    ok = True
    for n in [int(x) for x in args.sizes.split(",")]:
        samples = [W.uniform_points(1 + i, args.iterations, [-W.ENV_RAD] * 3, [W.ENV_RAD] * 3) for i in range(n)]
        run_lockstep(ctx, S, [s[:20] for s in samples], 20)   # warm-up of both forms' modules and buffers at this size
        run_serial(ctx, S, samples[:1], 20)
        best_a, best_b, med_b, ha, hb = np.inf, np.inf, None, set(), set()
        for _ in range(args.reps):
            sa, _, h = run_serial(ctx, S, samples, args.iterations)
            best_a = min(best_a, sa)
            ha.add(h)
            sb, mb, h = run_lockstep(ctx, S, samples, args.iterations)
            if sb < best_b:
                best_b, med_b = sb, mb
            hb.add(h)
        iters = n * args.iterations
        same = len(ha) == 1 and ha == hb
        ok &= same
        line = {"experiment": "lockstep_instances", "gpu": name, "power_limit": power, "instances": n,
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
