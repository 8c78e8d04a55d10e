"""Child process of tests/test_odom_stress.py::test_forced_tiled_and_voxel_sort_paths_reproduce_the_session.

SB_SORT_TILED (the tree build's sort skips the one-CTA shared-memory path) and SB_VOXEL_SORT (the voxel grid skips the
hashed path) are read once per process, so the session runs with both forced in a process of its own:
SB_SORT_TILED=1 SB_VOXEL_SORT=1 python odom_stress_worker.py <dir>.  <dir> holds two streams of frames, plain_scan_<i>.npy
(float32-born rows) and jitter_scan_<i>.npy (the same rows plus 1e-9-scale noise), and the parent's session bits of
each frame (<stream>_bits_<i>.npy, test_odom_session.frame_bits with every output).  Prints one marker line per check.
"""
import os
import sys


def usage(msg):
    print(f"odom_stress_worker: {msg}", file=sys.stderr)
    sys.exit(2)


def main(argv):
    if len(argv) != 2:
        usage("usage: SB_SORT_TILED=1 SB_VOXEL_SORT=1 python odom_stress_worker.py <dir>")
    if os.environ.get("SB_SORT_TILED") != "1" or os.environ.get("SB_VOXEL_SORT") != "1":
        usage("needs SB_SORT_TILED=1 SB_VOXEL_SORT=1 in the environment")
    d = argv[1]
    names = os.listdir(d) if os.path.isdir(d) else []
    n = len([f for f in names if f.startswith("plain_scan_")])
    if n == 0:
        usage(f"no frames in {d}")

    import numpy as np
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, here)
    sys.path.insert(0, os.path.join(os.path.dirname(here), "lidar-slam-from-scratch_b200", "python"))
    import slam_b200
    from test_odom_session import frame_bits, same_bits
    from test_odom_stress import ALL, assert_matches_per_call, per_call_loop

    eng = slam_b200.Engine(0)
    for stream in ("plain", "jitter"):
        scans = [np.load(os.path.join(d, f"{stream}_scan_{i}.npy")) for i in range(n)]
        want = [np.load(os.path.join(d, f"{stream}_bits_{i}.npy")) for i in range(n)]
        odom = slam_b200.Odometry(eng)
        frames = []
        for i, s in enumerate(scans):
            frames.append(odom.push(s, i, **ALL))
            assert eng.last_voxel_path == 2, (stream, i)
        odom.close()
        for i, (f, w) in enumerate(zip(frames, want)):
            assert same_bits(frame_bits(f), w), (stream, i)
        assert_matches_per_call(frames, per_call_loop(eng, scans), stream)
        print(f"FORCED_SORT_{stream.upper()} {n} frames identical to the default process and the per-call loop, "
              f"{min(f.n_points for f in frames)}..{max(f.n_points for f in frames)} rows", flush=True)
    eng.close()
    print("ODOM_STRESS_WORKER_OK", flush=True)


if __name__ == "__main__":
    main(sys.argv)
