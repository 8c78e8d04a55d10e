"""Streaming odometry: the node's per-call loop (scripts/stream_latency.py's process_frames: voxel_downsample,
icp_point_to_plane, transform_clouds, addFrame, detect() every tenth frame after frame 50) against the streaming session
(slam_b200.Odometry: one push per frame, previous frame kept on the device) on the same frames, in one process.  After a
warm-up run of each, the two paths alternate `--reps` times.  Prints one JSON line: per path ms/frame mean / p50 / p99
(the mean over repetitions of each repetition's figure, and every repetition), launches per frame, and the card it ran
on (name and power limit, read with nvidia-smi's read-only query).  The per-call loop gets the world-frame cloud as fp64
rows (transform_clouds, as stream_latency.py does); the session returns the downsampled rows and the float32 PointCloud2
payload.

  python scripts/odom_session_bench.py [--frames 120] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "lidar-slam-from-scratch_b200", "python"))
sys.dont_write_bytecode = True


def session_frames(eng, slam_b200, scans, voxel=0.5, skip=10):
    """The same loop through one Odometry session: every frame is added to the detector (as process_frames does,
    frame 0 included), detect() on the node's schedule, the world-frame cloud (PointCloud2 float32) and the downsampled
    rows come back every frame.  Frames up to `skip` are warm-up."""
    det = slam_b200.LoopClosureDetector(eng)
    odom = slam_b200.Odometry(eng, voxel=voxel, loop=det)
    odom.reserve(max(len(s) for s in scans))
    total = []
    odom.push(scans[0], 0, want_cloud=True, want_world_f32=True)
    launches0 = eng.launch_count
    for i in range(1, len(scans)):
        t0 = time.perf_counter()
        odom.push(scans[i], i, detect=(i % 10 == 0 and i > 50), want_cloud=True, want_world_f32=True)
        t1 = time.perf_counter()
        if i > skip:
            total.append(t1 - t0)
    launches = eng.launch_count - launches0
    odom.close()
    det.close()
    t = np.array(total) * 1e3
    return {"ms": t, "launches_per_frame": launches / (len(scans) - 1)}


def rep_stats(ms):
    """ms/frame of one repetition, computed as stream_latency.process_frames computes its own."""
    return {"ms_per_frame_mean": float(ms.mean()), "p50": float(np.percentile(ms, 50)), "p99": float(np.percentile(ms, 99)),
            "max": float(ms.max())}


def summary(reps, launches, frames):
    """Per path: the mean over repetitions of each per-repetition figure, and the repetitions themselves."""
    keys = ("ms_per_frame_mean", "p50", "p99", "max")
    out = {k: float(np.mean([r[k] for r in reps])) for k in keys}
    out["reps"] = [{k: round(r[k], 4) for k in keys} for r in reps]
    out["frames_timed_per_rep"] = frames
    out["launches_per_frame"] = launches
    return out


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[0].split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"gpu": f"unknown ({e})", "power_limit": "unknown"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=120)
    ap.add_argument("--voxel", type=float, default=0.5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import bench
    import slam_b200
    import stream_latency
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib

    syn = oracle_lib.Synth()  # pose / scene tables (host side of the raycaster)
    world = bench.make_world(syn)
    F = args.frames
    poses = bench.make_poses(syn, F + 1)
    eng = slam_b200.Engine(0)
    rays = bench.SENSOR["beams"] * bench.SENSOR["azimuth_steps"]
    d_raw = torch.empty((F + 1) * rays * 3, dtype=torch.float64, device="cuda")
    off = eng.synth_scans_dev(bench.SENSOR, world, poses, 1000, d_raw.data_ptr())
    h = d_raw[:int(off[-1]) * 3].cpu().numpy().reshape(-1, 3)
    del d_raw
    scans = [np.ascontiguousarray(h[off[i]:off[i + 1]]) for i in range(F + 1)]

    per_call = lambda: stream_latency.process_frames(eng, slam_b200, scans, args.voxel)  # noqa: E731
    session = lambda: session_frames(eng, slam_b200, scans, args.voxel)  # noqa: E731
    per_call(), session()   # warm-up: allocations, graphs, pools
    reps = {"per_call": [], "session": []}
    launches, frames, split = {}, {}, None
    for _ in range(args.reps):
        r = per_call()
        reps["per_call"].append(r)
        launches["per_call"], frames["per_call"], split = r["launches_per_frame"], r["frames"], r["split_ms_mean"]
        s = session()
        reps["session"].append(rep_stats(s["ms"]))
        launches["session"], frames["session"] = s["launches_per_frame"], int(len(s["ms"]))
    out = {"workload": f"process_frame loop (slam_node.cpp:118-175), {F + 1} frames of bench.py's sensor, voxel "
                       f"{args.voxel}, detect() every tenth frame after 50, frames 1..10 untimed; the two paths "
                       f"alternated {args.reps}x in one process after one warm-up run each",
           **card(),
           "per_call": summary(reps["per_call"], launches["per_call"], frames["per_call"]),
           "session": summary(reps["session"], launches["session"], frames["session"]),
           "per_call_split_ms_mean_last_rep": split}
    out["speedup_mean"] = out["per_call"]["ms_per_frame_mean"] / out["session"]["ms_per_frame_mean"]
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    eng.close()


if __name__ == "__main__":
    main()
