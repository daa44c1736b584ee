#!/usr/bin/env python
"""A/B of library builds on every path of the sphere-world collision kernels: the per-call batch check (thread-per-edge
and two-stage), the resident check and the obstacle-add sweep (item grid, two-stage, thread-per-item, node-centric with
statistics), the remove sweep, the tiled small-batch check and the point check.

    python scripts/exp_collision_paths.py LIB_A LIB_B [--reps 3]

runs one worker process per build and repetition, alternating the builds (RRTQX_B200_LIB selects the build).  Every
row prints the median of the library's phase times (CUDA events; L2 overwritten by a 256 MiB memset before each call)
and a hash of the returned flags or id lists.  The rows use the C3 edge set of bench.py (1M-node C2 tree, edges within
0.5346, parent edges) and the 256 C3 spheres; "small" is the C3-style graph of the nodes with x below the 9% quantile
(same density, under 2^20 items: its add sweep takes the thread-per-item path by default)."""
import hashlib
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SWITCHES = ("RRTQX_COVER_MIN_ITEMS", "RRTQX_NO_ITEM_GRID", "RRTQX_EDGE_NO_QUEUE")


def worker():
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    import bench
    from rrtqx_3d_b200 import _abi as A
    from rrtqx_3d_b200 import workloads as W
    from rrtqx_3d_b200.device import (Context, DeviceTree, EdgeSet, SphereSet, SweepResult, edge_check_batch,
                                      node_check_batch)

    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = Context(0, stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    pts, _, _ = W.c2_workload(1_000_000, 1)
    tree = DeviceTree(ctx, 3)
    tree.insert_batch(pts)
    src, dst, parent = bench.build_c3_edges(tree, pts, 0.5346)
    E = EdgeSet(tree)
    E.upload(src, dst, parent)
    small_pts = np.ascontiguousarray(pts[pts[:, 0] < np.quantile(pts[:, 0], 0.09)])
    tree_s = DeviceTree(ctx, 3)
    tree_s.insert_batch(small_pts)
    s_src, s_dst, s_parent = bench.build_c3_edges(tree_s, small_pts, 0.5346)
    E_s = EdgeSet(tree_s)
    E_s.upload(s_src, s_dst, s_parent)
    centers, radii = W.c3_obstacles(256)
    S = SphereSet(ctx, centers, radii)
    ids = np.arange(256, dtype=np.int32)
    sres = SweepResult(ctx)
    dsrc, ddst = torch.from_numpy(src).cuda(), torch.from_numpy(dst).cuda()
    dflag = torch.empty(len(src), dtype=torch.uint8, device="cuda")
    edge_dist_inf = np.zeros(len(src), dtype=np.uint8)
    node_pts = W.uniform_points(11, 100_000, [-W.ENV_RAD] * 3, [W.ENV_RAD] * 3)

    def h(*arrays):
        d = hashlib.sha1()
        for a in arrays:
            d.update(np.ascontiguousarray(a).tobytes())
        return d.hexdigest()[:12]

    def sweep_hash():
        e, n = sres.fetch()
        return h(np.sort(e), np.sort(n))

    def tune(**env):
        for k in SWITCHES:
            os.environ.pop(k, None)
        os.environ.update({k: str(v) for k, v in env.items()})
        ctx.reload_tuning()

    def row(name, fn, phase, digest, reps=10):
        ms = []
        for it in range(3 + reps):
            flush.zero_()
            fn()
            if it >= 3:
                ms.append(ctx.last_phase_ms(phase))
        print(f"ROW {name:44s} {np.median(ms):9.4f} ms  {digest()}", flush=True)

    def batch(n, fl):
        return lambda: edge_check_batch(tree, S, dsrc, ddst, W.ROBOT_RADIUS, flags=fl, n_edges=n, out=dflag)

    for env, tag in (({}, "thread-per-edge"), ({"RRTQX_COVER_MIN_ITEMS": 1}, "two-stage")):
        tune(**env)
        for n in (6_000, 200_000, 1_500_000):
            for fl in (0, A.CHECK_FMA_DOT):
                row(f"edge_check_batch {n} {tag} fma={fl}", batch(n, fl), "edge_check", lambda n=n: h(dflag[:n].cpu().numpy()))
    tune()
    row("edge_check_batch 2000 tiled", batch(2_000, 0), "edge_check", lambda: h(dflag[:2_000].cpu().numpy()))

    for env, tag in (({"RRTQX_NO_ITEM_GRID": 1}, "two-stage"),
                     ({"RRTQX_NO_ITEM_GRID": 1, "RRTQX_EDGE_NO_QUEUE": 1}, "no-queue"),
                     ({}, "item-grid")):
        tune(**env)
        for fl in (0, A.CHECK_FMA_DOT):
            row(f"edges_check full {tag} fma={fl}", lambda fl=fl: E.check_all(S, W.ROBOT_RADIUS, flags=fl, out=dflag.data_ptr()),
                "edges_check", lambda: h(dflag.cpu().numpy()))
            for k, obs in ((256, ids), (1, ids[7:8])):
                row(f"add_sweep full {k} {tag} fma={fl}", lambda obs=obs, fl=fl: E.add_sweep(S, obs, W.ROBOT_RADIUS, W.DELTA, flags=fl, result=sres),
                    "add_sweep", sweep_hash)
    for env, tag in (({"RRTQX_NO_ITEM_GRID": 1}, "thread-per-item"), ({}, "item-grid")):
        tune(**env)
        s_flag = torch.empty(len(s_src), dtype=torch.uint8, device="cuda")
        row(f"edges_check small {tag}", lambda: E_s.check_all(S, W.ROBOT_RADIUS, out=s_flag.data_ptr()), "edges_check",
            lambda: h(s_flag.cpu().numpy()))
        for fl in (0, A.CHECK_FMA_DOT):
            for k, obs in ((256, ids), (1, ids[7:8])):
                row(f"add_sweep small {k} {tag} fma={fl}", lambda obs=obs, fl=fl: E_s.add_sweep(S, obs, W.ROBOT_RADIUS, W.DELTA, flags=fl, result=sres),
                    "add_sweep", sweep_hash)
    tune()
    row("add_sweep full 256 statistics", lambda: E.add_sweep(S, ids, W.ROBOT_RADIUS, W.DELTA, flags=A.SWEEP_STATS, result=sres),
        "add_sweep", lambda: sweep_hash() + " " + h(np.array(sres.sizes())))
    E.add_sweep(S, ids, W.ROBOT_RADIUS, W.DELTA, result=sres)
    e_hit, _ = sres.fetch()
    edge_dist_inf[e_hit] = 1
    row("remove_sweep full", lambda: E.remove_sweep(S, 7, np.delete(ids, 7), edge_dist_inf, W.ROBOT_RADIUS, W.DELTA, result=sres),
        "remove_sweep", sweep_hash)
    out = {}

    def point_check():
        out["r"] = node_check_batch(ctx, S, node_pts, W.ROBOT_RADIUS)
    row("node_check 1e5 points", point_check, "node_check", lambda: h(*out["r"]))


def main():
    if sys.argv[1:2] == ["--worker"]:
        return worker()
    libs = [os.path.abspath(p) for p in sys.argv[1:3]]
    reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 3
    import torch
    props = torch.cuda.get_device_properties(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    print(f"card: {props.name} | nvidia-smi: {smi.stdout.strip()}", flush=True)
    for r in range(reps):
        for lib in libs:
            print(f"== rep {r} lib {lib}", flush=True)
            env = {k: v for k, v in os.environ.items() if k not in SWITCHES}
            env["RRTQX_B200_LIB"] = lib
            subprocess.run([sys.executable, os.path.abspath(__file__), "--worker"], env=env, check=True)


if __name__ == "__main__":
    main()
