"""Loop-closure rebuild of the node's map (slam_node.cpp:177-209): after PoseGraph::optimize every pose changes, and the
occupancy grid, the window of the last 20 world clouds and the global map (voxel 2 * voxel_size) are rebuilt.

  stateless  host clouds -> sb_occupancy_cells + sb_global_map_f32 + sb_transform_clouds_f32 (20-cloud window): every
             call uploads the clouds it needs
  map        sb_map_set_poses (poses only) + sb_map_occupancy_cells + sb_map_global_f32 + sb_map_world_f32

for F keyframes of bench.py's sensor (downsampled by a streaming session that also fills the map, SB_ODOM_ADD_MAP).
The two paths alternate `--reps` times after a warm-up of each, on the same corrected poses, and their outputs are
compared bit for bit.  It also times a push with and without the map add over the same frames.  Prints one JSON line:
ms mean / p50 / p99 per path, host-to-device bytes per rebuild, and the card (name, power limit).

  python scripts/map_bench.py [--frames 1000,4541] [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "lidar-slam-from-scratch_b200", "python"))
sys.dont_write_bytecode = True

WINDOW = 20


def stats(ms):
    ms = np.asarray(ms)
    return {"ms_mean": float(ms.mean()), "p50": float(np.percentile(ms, 50)), "p99": float(np.percentile(ms, 99)),
            "reps": [round(float(v), 3) for v in ms]}


def keyframes(eng, slam_b200, torch, bench, syn, F, voxel, chunk=250):
    """The session over F frames (raw scans made on the device chunk by chunk), adding every frame to a map; returns
    the map, the downsampled clouds, the poses and the push times with the map add."""
    world = bench.make_world(syn)
    poses = bench.make_poses(syn, F)
    rays = bench.SENSOR["beams"] * bench.SENSOR["azimuth_steps"]
    m = slam_b200.Map(eng)
    odom = slam_b200.Odometry(eng, voxel=voxel, map=m)
    odom.reserve(rays)
    clouds, Ts = [], []
    d_raw = torch.empty(chunk * rays * 3, dtype=torch.float64, device="cuda")
    for c0 in range(0, F, chunk):
        n = min(chunk, F - c0)
        off = eng.synth_scans_dev(bench.SENSOR, world, poses[c0:c0 + n], 1000 + c0, d_raw.data_ptr())
        h = d_raw[:int(off[-1]) * 3].cpu().numpy().reshape(-1, 3)
        for i in range(n):
            f = odom.push(np.ascontiguousarray(h[off[i]:off[i + 1]]), c0 + i, want_cloud=True)
            clouds.append(f.cloud if f.state != slam_b200.ODOM_SKIPPED else np.zeros((0, 3)))
            Ts.append(f.pose)
    odom.close()
    return m, clouds, np.stack(Ts)


def push_cost(eng, slam_b200, scans, voxel, reps):
    """ms per push over the same frames, with and without the map add, alternating."""
    out = {"without_map": [], "with_map": []}
    for r in range(reps + 1):
        for kind in ("without_map", "with_map"):
            m = slam_b200.Map(eng) if kind == "with_map" else None
            odom = slam_b200.Odometry(eng, voxel=voxel, map=m)
            odom.reserve(max(len(s) for s in scans))
            if m is not None:
                m.reserve(len(scans), 12_000 * len(scans), 50_000 * len(scans))
            t = []
            for i, s in enumerate(scans):
                t0 = time.perf_counter()
                odom.push(s, i)
                t.append(time.perf_counter() - t0)
            odom.close()
            if m is not None:
                m.close()
            if r > 0:
                out[kind].append(float(np.mean(t[10:]) * 1e3))
    return {k: stats(v) for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", default="1000,4541")
    ap.add_argument("--voxel", type=float, default=0.5)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import bench
    import slam_b200
    from odom_session_bench import card
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib

    if not torch.cuda.is_available():
        raise SystemExit("map_bench.py measures on the GPU; no CUDA device is visible")
    syn = oracle_lib.Synth()
    eng = slam_b200.Engine(0)
    sizes = [int(x) for x in args.frames.split(",")]
    full, clouds, poses = keyframes(eng, slam_b200, torch, bench, syn, max(sizes), args.voxel)
    rng = np.random.default_rng(0)
    result = {"workload": f"loop-closure rebuild of the map (slam_node.cpp:177-209): occupancy cells, the last {WINDOW} "
                          f"world clouds as float32, the global map at voxel {2 * args.voxel} as float32; keyframes of "
                          f"bench.py's sensor downsampled at {args.voxel}; {args.reps} alternating repetitions after "
                          f"one warm-up of each path; host clock around calls that end in a synchronise",
              **card(), "rebuild": {}}
    for F in sizes:
        cl, Ts = clouds[:F], poses[:F]
        if F == len(clouds):
            m = full
        else:
            m = slam_b200.Map(eng)
            for c, P in zip(cl, Ts):
                m.add(c, P)
        off = np.r_[0, np.cumsum([len(c) for c in cl])].astype(np.int64)
        pts = np.concatenate(cl)
        woff = off[F - WINDOW:] - off[F - WINDOW]
        wpts = pts[off[F - WINDOW]:]
        times = {"stateless": [], "map": []}
        outs = {}
        for r in range(args.reps + 1):
            D = np.eye(4)
            D[:3, 3] = rng.uniform(-0.5, 0.5, 3)
            new = np.einsum("ij,fjk->fik", D, Ts)   # a correction of every pose
            t0 = time.perf_counter()
            a = (eng.occupancy_cells(pts, off, new), eng.global_map_f32(pts, off, new, 2 * args.voxel),
                 eng.transform_clouds_f32(wpts, woff, new[F - WINDOW:]))
            t1 = time.perf_counter()
            m.set_poses(new)
            b = (m.occupancy_cells(), m.global_map(2 * args.voxel, f32=True), m.world_f32(F - WINDOW, WINDOW))
            t2 = time.perf_counter()
            if r > 0:
                times["stateless"].append((t1 - t0) * 1e3)
                times["map"].append((t2 - t1) * 1e3)
            same = (a[0][1] == b[0][1] and np.array_equal(a[0][0], b[0][0]) and
                    a[1].tobytes() == b[1].tobytes() and a[2].tobytes() == b[2].tobytes())
            if not same:
                raise SystemExit(f"F={F}: the map's outputs differ from the stateless calls")
            outs = {"cells": int(b[0][1]), "global_map_rows": int(len(b[1])), "window_rows": int(len(b[2]))}
        rows = int(off[-1])
        h2d_stateless = 2 * (24 * rows + 8 * (F + 1) + 128 * F) + 24 * len(wpts) + 8 * (WINDOW + 1) + 128 * WINDOW
        result["rebuild"][str(F)] = {"entries": F, "rows": rows, **outs, "bit_identical": True,
                                     "stateless": stats(times["stateless"]), "map": stats(times["map"]),
                                     "h2d_bytes_stateless": h2d_stateless, "h2d_bytes_map": 128 * F,
                                     "speedup_mean": float(np.mean(times["stateless"]) / np.mean(times["map"]))}
        if m is not full:
            m.close()
    # per-frame cost of the add inside the session, on the first 300 frames (scans regenerated on the device)
    n = min(300, max(sizes))
    world = bench.make_world(syn)
    ps = bench.make_poses(syn, n)
    rays = bench.SENSOR["beams"] * bench.SENSOR["azimuth_steps"]
    d_raw = torch.empty(n * rays * 3, dtype=torch.float64, device="cuda")
    off = eng.synth_scans_dev(bench.SENSOR, world, ps, 1000, d_raw.data_ptr())
    h = d_raw[:int(off[-1]) * 3].cpu().numpy().reshape(-1, 3)
    del d_raw
    scans = [np.ascontiguousarray(h[off[i]:off[i + 1]]) for i in range(n)]
    result["push_ms_per_frame"] = {"frames": n, "frames_timed": n - 10, **push_cost(eng, slam_b200, scans, args.voxel,
                                                                                   args.reps)}
    full.close()
    eng.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
