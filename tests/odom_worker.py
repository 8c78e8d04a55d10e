"""Child process of tests/test_odom_session.py::test_failed_pushes_leave_the_session_unchanged.

Failed pushes must leave a streaming session exactly as it was.  The checks run in a process of their own so that an
unexpected device fault cannot poison the test session's shared engine: python odom_worker.py <dir>, where <dir> holds
the parent's frames (scan_<i>.npy).  Prints one marker line per check.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "lidar-slam-from-scratch_b200", "python"))

import slam_b200  # noqa: E402
from test_odom_session import frame_bits, same_bits  # noqa: E402


def expect_status(call, status):
    try:
        call()
    except slam_b200.SlamB200Error as e:
        assert e.status == status, e
        return
    raise AssertionError(f"no error, expected status {status}")


def run(sess, scans, frames, **kw):
    return [frame_bits(sess.push(scans[i], i, want_cloud=True, want_world_f32=True, want_desc=True, **kw))
            for i in frames]


def main(d):
    n = len([f for f in os.listdir(d) if f.startswith("scan_")])
    scans = [np.load(os.path.join(d, f"scan_{i}.npy")) for i in range(n)]
    eng = slam_b200.Engine(0)
    frames = range(n)
    cut = n // 2

    def detector(**kw):
        return slam_b200.LoopClosureDetector(eng, frame_gap=2, sc_distance_threshold=1e300, **kw)

    # the reference: a session (min_points 0, detector attached) that never sees a bad call
    det_a = detector()
    a = slam_b200.Odometry(eng, min_points=0, loop=det_a)
    want = run(a, scans, frames)
    want_cand = det_a.candidates_local()

    # 1. a NaN row (SB_ERR_RANGE, found by the voxel grid) and an empty frame with min_points 0 (SB_ERR_EMPTY), twice
    # each, half way through the sequence
    det_b = detector()
    b = slam_b200.Odometry(eng, min_points=0, loop=det_b)
    got = run(b, scans, range(cut))
    size = det_b.size()
    bad = scans[cut].copy()
    bad[len(bad) // 3] = np.nan
    for _ in range(2):
        expect_status(lambda: b.push(bad, cut, detect=True), 5)
        expect_status(lambda: b.push(np.empty((0, 3)), cut), 2)
        expect_status(lambda: b.push(bad.astype(np.float32), cut), 5)
    assert det_b.size() == size
    got += run(b, scans, range(cut, n))
    assert all(same_bits(g, w) for g, w in zip(got, want))
    got_cand = det_b.candidates_local()
    assert all(same_bits(x, y) for x, y in zip(got_cand, want_cand))
    print("RANGE_AND_EMPTY unchanged", flush=True)

    # 2. SB_ODOM_DETECT without a detector, and with a world-2 detector
    c = slam_b200.Odometry(eng, min_points=0)
    det_w2 = detector(rank=0, world=2)
    d2 = slam_b200.Odometry(eng, min_points=0, loop=det_w2)
    got_c, got_d = run(c, scans, range(cut)), run(d2, scans, range(cut))
    expect_status(lambda: c.push(scans[cut], cut, detect=True), 1)
    expect_status(lambda: d2.push(scans[cut], cut, detect=True), 1)
    got_c += run(c, scans, range(cut, n))
    got_d += run(d2, scans, range(cut, n))
    assert all(same_bits(g, w) for g, w in zip(got_c, want))
    assert all(same_bits(g, w) for g, w in zip(got_d, want))
    assert det_w2.size() == n
    print("INVALID_ARG unchanged", flush=True)
    for s in (a, b, c, d2):
        s.close()
    for x in (det_a, det_b, det_w2):
        x.close()
    eng.close()
    print("ODOM_WORKER_OK", flush=True)


if __name__ == "__main__":
    main(sys.argv[1])
