"""Many live streams on one GPU: one slam_b200.push_many call per frame step (sb_odom_push_many: one voxel grid, one
index build, one ICP batch for all streams) against N consecutive single pushes (Odometry.push, sb_odom_push) of the
same frames, in one process.  N streams on N different scenes (bench.py's C5 scene recipe, seed 100 + s), each driving
its own straight trajectory, scanned with bench.py's sensor (~119 k rows per scan), voxel 0.5; the downsampled rows and
the world-frame float32 cloud come back every frame, as in scripts/odom_session_bench.py.  Every path runs `--frames`
frame steps per stream with fresh sessions, the first 10 untimed; after one warm-up run of each path the two paths
alternate `--reps` times.  The scans of a step are generated on the device and copied to host memory before the step
(untimed); the calls are timed with the host clock and return after their final synchronise.

Writes one JSON file under --out-dir (and prints it): per N and path the aggregate frames/s, ms per call (one call = one
push_many, or N single pushes) mean / p50 / p99 over all timed steps of all repetitions, launches per call, and the card
(name, power limit, max SM clock, read with nvidia-smi's read-only query in the same run).

  python scripts/odom_many_bench.py [--streams 1,8,32,128] [--frames 40] [--reps 3] [--out-dir DIR]
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
sys.path.insert(0, os.path.join(ROOT, "lidar-slam-from-scratch_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True

SKIP = 10


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power, clock = [x.strip() for x in out[0].split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"gpu": f"unknown ({e})", "power_limit": "unknown", "max_sm_clock": "unknown"}


class Frames:
    """Frame step i of N streams, raycast on the device (stream s: scene 100 + s, lateral offset, noise seed)."""

    def __init__(self, eng, syn, bench, n):
        import torch
        self.eng, self.bench, self.n = eng, bench, n
        self.worlds = [bench.c5_scene(syn, s) for s in range(n)]
        self.syn = syn
        rays = bench.SENSOR["beams"] * bench.SENSOR["azimuth_steps"]
        self.d = torch.empty(rays * 3, dtype=torch.float64, device="cuda")
        self.cache = {}

    def step(self, i):
        if i in self.cache:
            return self.cache[i]
        out = []
        for s in range(self.n):
            pose = np.array([self.syn.pose(0, 0.0, 1.0 * i - 20.0, 0.5 * ((s % 5) - 2))])
            off = self.eng.synth_scans_dev(self.bench.SENSOR, self.worlds[s], pose, 700000 + 1000 * s + i, self.d.data_ptr())
            self.eng.synchronize()
            out.append(self.d[:int(off[-1]) * 3].cpu().numpy().reshape(-1, 3).copy())
        if self.n <= 32:   # <= 3.7 GB of rows for 40 steps: kept; larger N are raycast again for each run
            self.cache[i] = out
        return out


def run(eng, slam_b200, frames, n, n_frames, many, voxel):
    sess = [slam_b200.Odometry(eng, voxel=voxel) for _ in range(n)]
    ms, launches = [], []
    for i in range(n_frames):
        fr = frames.step(i)
        l0 = eng.launch_count
        t0 = time.perf_counter()
        if many:
            slam_b200.push_many(sess, fr, i, want_cloud=True, want_world_f32=True)
        else:
            for o, f in zip(sess, fr):
                o.push(f, i, want_cloud=True, want_world_f32=True)
        t1 = time.perf_counter()
        if i >= SKIP:
            ms.append((t1 - t0) * 1e3)
            launches.append(eng.launch_count - l0)
    for o in sess:
        o.close()
    return ms, launches


def stats(ms, launches, n):
    a = np.array(ms)
    return {"frames_per_s": float(n * 1e3 / a.mean()), "ms_per_call_mean": float(a.mean()),
            "ms_per_call_p50": float(np.percentile(a, 50)), "ms_per_call_p99": float(np.percentile(a, 99)),
            "ms_per_frame_mean": float(a.mean() / n), "launches_per_call": float(np.mean(launches)), "calls_timed": len(a)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", default="1,8,32,128")
    ap.add_argument("--frames", type=int, default=40)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--voxel", type=float, default=0.5)
    ap.add_argument("--out-dir", default=".")
    args = ap.parse_args()
    import bench
    import oracle_lib
    import slam_b200
    syn = oracle_lib.Synth()
    eng = slam_b200.Engine(0)
    result = {"workload": f"N streams on N scenes, bench.py's sensor, voxel {args.voxel}, {args.frames} frame steps per "
                          f"stream with the first {SKIP} untimed; one push_many per step against N single pushes, "
                          f"alternated {args.reps}x after one warm-up run each",
              **card(), "streams": {}}
    for n in [int(x) for x in args.streams.split(",")]:
        frames = Frames(eng, syn, bench, n)
        warm = min(args.frames, SKIP + 2)
        run(eng, slam_b200, frames, n, warm, True, args.voxel)
        run(eng, slam_b200, frames, n, warm, False, args.voxel)
        acc = {"many": ([], []), "single": ([], [])}
        for _ in range(args.reps):
            for path in ("many", "single"):
                ms, la = run(eng, slam_b200, frames, n, args.frames, path == "many", args.voxel)
                acc[path][0].extend(ms)
                acc[path][1].extend(la)
        r = {p: stats(acc[p][0], acc[p][1], n) for p in acc}
        r["speedup_frames_per_s"] = r["many"]["frames_per_s"] / r["single"]["frames_per_s"]
        result["streams"][str(n)] = r
        print(f"[odom_many_bench] N={n}: many {r['many']['frames_per_s']:.0f} frames/s, single "
              f"{r['single']['frames_per_s']:.0f} frames/s, x{r['speedup_frames_per_s']:.2f}", flush=True)
    eng.close()
    os.makedirs(args.out_dir, exist_ok=True)
    line = json.dumps(result)
    with open(os.path.join(args.out_dir, "odom_many_bench.json"), "w") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
