"""Streaming odometry session (sb_odom_*, slam_b200.Odometry, slam::b200::Odometry): SlamNode::process_frame
(slam_node.cpp:118-175) one scan per call with the previous frame kept on the device, checked bit for bit against the
node's per-call loop over the single-call entry points (voxel_downsample, icp_point_to_plane, sb_odometry_poses,
transform_clouds_f32, sc_compute, LoopClosureDetector addFrame / detect_batch).  The per-call loop itself is checked
against the oracle by test_scale_parity.py::test_streaming_sequence_with_loop_closures_matches_oracle.
"""
import ctypes as C
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "lidar-slam-from-scratch_b200", "python"))
import slam_b200  # noqa: E402

# streaming sequence: a loop of 2 pi 10.5 m = 66 m driven at 1 m per frame, so frames 66.. revisit frames 0..; with the
# node's frame gap of 50 the detect() of frame 70 finds its loop closures among frames 0..20 (noise seeds 500 + i)
STREAM_RADIUS, STREAM_SCENE, STREAM_FRAMES = 10.5, 3, 78
VOXEL = 0.5


def cores():
    return os.cpu_count() or 1


def same_bits(a, b):
    a, b = np.ascontiguousarray(a, dtype=np.float64), np.ascontiguousarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def icp_bits(r):
    """Every field of an ICPResult as float64: T[16], final_error, converged, num_iterations, status, history."""
    return np.concatenate([r.transformation.reshape(16), [r.final_error, r.converged, r.num_iterations, r.status,
                                                          len(r.error_history)], r.error_history])


def frame_bits(f):
    """Everything an OdomFrame carries (outputs that were not asked for count as empty)."""
    parts = [[f.frame_idx, f.state, f.n_points, f.n_loops], f.pose.reshape(16)]
    parts.append(icp_bits(f.icp) if f.icp is not None else [])
    for a in (f.cloud, f.world_f32, f.desc):
        parts.append([] if a is None else np.asarray(a, dtype=np.float64).reshape(-1))
    for r in f.loops:
        parts.append(loop_bits(r))
    return np.concatenate([np.asarray(p, dtype=np.float64).reshape(-1) for p in parts])


def loop_bits(r):
    return np.concatenate([[r["query_frame"], r["match_frame"], r["scan_context_distance"], r["icp_fitness"]],
                           np.asarray(r["transform"]).reshape(16)])


def host_pose_product(P, D):
    """Transformation::operator* (types.hpp:118-125) as sb_odometry_poses forms it: k ascending from 0.0."""
    out = np.empty((4, 4))
    for i in range(4):
        for j in range(4):
            acc = 0.0
            for k in range(4):
                acc += float(P[i, k]) * float(D[k, j])
            out[i, j] = acc
    return out


def node_detects(i):
    return i % 10 == 0 and i > 50      # slam_node.cpp:160


def odom_config_probe():
    prog = r'''
#include <stdio.h>
#include <stddef.h>
#include "slam_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(sb_odom_config), offsetof(sb_odom_config, max_error),
         offsetof(sb_odom_config, icp), offsetof(sb_odom_config, initial_pose), sizeof(sb_odom_frame),
         offsetof(sb_odom_frame, n_points), offsetof(sb_odom_frame, pose), offsetof(sb_odom_frame, icp),
         offsetof(sb_odom_frame, n_loops));
  return 0; }
'''
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "t.c")
        with open(src, "w") as fh:
            fh.write(prog)
        exe = os.path.join(d, "t")
        subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        return [int(x) for x in subprocess.check_output([exe]).split()]


# ------------------------------------------------------------------ CPU
def test_odom_ctypes_layout_matches_header():
    Cfg, Fr = slam_b200.OdomConfigC, slam_b200.OdomFrameC
    want = [C.sizeof(Cfg), Cfg.max_error.offset, Cfg.icp.offset, Cfg.initial_pose.offset, C.sizeof(Fr),
            Fr.n_points.offset, Fr.pose.offset, Fr.icp.offset, Fr.n_loops.offset]
    assert odom_config_probe() == want


def test_odom_defaults_match_the_node():
    lib = slam_b200.load_library()
    cfg = slam_b200.OdomConfigC()
    lib.sb_default_odom_config(C.byref(cfg))
    assert (cfg.voxel, cfg.min_points, cfg.max_error) == (0.5, 1000, 1.0)   # slam_node voxel_size, slam_node.hpp:29, :139
    icp = slam_b200.ICPConfigC()
    lib.sb_default_icp_config(C.byref(icp))
    assert bytes(cfg.icp) == bytes(icp)
    assert list(cfg.initial_pose) == [1.0 if i % 5 == 0 else 0.0 for i in range(16)]


def test_odom_needs_a_device_and_a_context():
    lib = slam_b200.load_library()
    cfg = slam_b200.OdomConfigC()
    lib.sb_default_odom_config(C.byref(cfg))
    h = C.c_void_p()
    assert lib.sb_odom_create(None, C.byref(cfg), None, C.byref(h)) == 1     # SB_ERR_INVALID_ARG
    assert lib.sb_odom_push(None, None, 0, 0, 0, None, None, None, None, None, 0) == 1
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(slam_b200.SlamB200Error) as e:
        slam_b200.Odometry(slam_b200.Engine(0))
    assert e.value.status == 4   # SB_ERR_NO_DEVICE: there is no CPU fallback


def build_mirror_test(out_dir):
    """tests/cpp/odom_session_test.cpp over the mirror headers, linked like tests/cpp/build.sh links host_api_test."""
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import oracle_lib
    oracle_lib.Synth()  # builds libsynth.so if needed
    lib = os.path.join(ROOT, "lidar-slam-from-scratch_b200")
    exe = os.path.join(out_dir, "odom_session_test")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-Wno-unused-function", "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(lib, "host"), os.path.join(ROOT, "tests", "cpp", "odom_session_test.cpp"),
                           "-o", exe, "-L" + lib, "-lslam_b200", "-L" + os.path.join(ROOT, "synth"), "-lsynth",
                           "-Wl,-rpath," + lib, "-Wl,-rpath," + os.path.join(ROOT, "synth")])
    return exe


def test_mirror_odometry_compiles():
    with tempfile.TemporaryDirectory() as d:
        assert os.path.exists(build_mirror_test(d))


# ------------------------------------------------------------------ GPU: the streaming sequence, per call and per session
@pytest.fixture(scope="module")
def stream_scans(synth):
    sys.path.insert(0, ROOT)
    import bench
    world = synth.scene(STREAM_SCENE, n_boxes=400, path_kind=1, radius=STREAM_RADIUS)
    return [synth.scan(bench.SENSOR, world, synth.pose(1, STREAM_RADIUS, float(i)), 500 + i, threads=cores())
            for i in range(STREAM_FRAMES)]


def loop_detector(engine, **kw):
    return slam_b200.LoopClosureDetector(engine, frame_gap=50, sc_distance_threshold=0.25, icp_fitness_threshold=0.3,
                                         max_candidates=3, **kw)


@pytest.fixture(scope="module")
def per_call(engine, stream_scans):
    """The node's loop over the single-call entry points (as in test_scale_parity's streaming test), with every
    output the session gives; launches per frame counted over the node's own calls."""
    cfg = engine.icp_config()
    det = loop_detector(engine)
    out = dict(clouds=[], icp=[None], world=[], desc=[], loops={}, launches=[])
    for i, scan in enumerate(stream_scans):
        l0 = engine.launch_count
        cur = engine.voxel_downsample(scan, VOXEL)
        if i > 0:
            out["icp"].append(engine.icp_point_to_plane(cur, out["clouds"][-1], cfg))
        det.addFrame(cur, i)
        if node_detects(i):
            out["loops"][i] = det.detect_batch([det.size() - 1])[0]
        out["launches"].append(engine.launch_count - l0)
        out["clouds"].append(cur)
        out["desc"].append(engine.sc_compute(cur))
    rec = np.zeros(STREAM_FRAMES - 1, dtype=slam_b200.ICP_DTYPE)
    for k, r in enumerate(out["icp"][1:]):
        rec[k]["transformation"] = r.transformation.reshape(16)
        rec[k]["final_error"], rec[k]["converged"], rec[k]["num_iterations"] = r.final_error, r.converged, r.num_iterations
        rec[k]["status"], rec[k]["history_len"] = r.status, len(r.error_history)
        rec[k]["error_history"][:len(r.error_history)] = r.error_history
    out["poses"] = engine.odometry_poses(slam_b200.ICPResultBatch(rec), max_error=1.0)
    for i, cur in enumerate(out["clouds"]):
        l0 = engine.launch_count
        out["world"].append(engine.transform_clouds_f32(cur, np.array([0, len(cur)], dtype=np.int64), out["poses"][i][None]))
        out["launches"][i] += engine.launch_count - l0   # publish_current_scan is part of the node's frame
    out["detector"] = det
    return out


@pytest.fixture(scope="module")
def session_run(engine, stream_scans):
    det = loop_detector(engine)
    odom = slam_b200.Odometry(engine, loop=det)
    frames, launches = [], []
    for i, scan in enumerate(stream_scans):
        l0 = engine.launch_count
        frames.append(odom.push(scan, i, add_frame=True, detect=node_detects(i), want_cloud=True, want_world_f32=True,
                                want_desc=True))
        launches.append(engine.launch_count - l0)
    odom.close()
    return dict(frames=frames, launches=launches, detector=det)


@pytest.mark.gpu
def test_session_matches_the_per_call_loop_bit_for_bit(per_call, session_run):
    accepted = 0
    for i, f in enumerate(session_run["frames"]):
        assert f.frame_idx == i
        assert f.state == (slam_b200.ODOM_FIRST if i == 0 else slam_b200.ODOM_REGISTERED), i
        assert f.n_points == len(per_call["clouds"][i])
        assert same_bits(f.cloud, per_call["clouds"][i]), i
        if i > 0:
            assert same_bits(icp_bits(f.icp), icp_bits(per_call["icp"][i])), i
        assert same_bits(f.pose, per_call["poses"][i]), i
        assert np.array_equal(f.world_f32.view(np.uint32), per_call["world"][i].view(np.uint32)), i
        assert same_bits(f.desc, per_call["desc"][i]), i
        if node_detects(i):
            want = per_call["loops"][i]
            assert f.n_loops == len(want) == len(f.loops), i
            for a, b in zip(f.loops, want):
                assert same_bits(loop_bits(a), loop_bits(b)), i
            accepted += len(want)
        else:
            assert f.n_loops == 0 and f.loops == []
    assert session_run["detector"].size() == per_call["detector"].size() == STREAM_FRAMES
    assert all(same_bits(a, b) for a, b in zip(session_run["detector"].candidates_local(),
                                               per_call["detector"].candidates_local()))
    assert accepted >= 1, "the path revisits its start: detect() must accept a loop closure"
    print(f"[odom] {STREAM_FRAMES} frames bit-identical to the per-call loop, {accepted} accepted loop closures")


@pytest.mark.gpu
def test_session_launches_fewer_kernels_per_frame(per_call, session_run):
    a = np.array(session_run["launches"][10:], dtype=np.float64)
    b = np.array(per_call["launches"][10:], dtype=np.float64)
    assert a.mean() < b.mean(), (a.mean(), b.mean())
    print(f"[odom] launches/frame over frames 10..{STREAM_FRAMES - 1}: session {a.mean():.1f}, per call {b.mean():.1f}")


@pytest.mark.gpu
def test_float32_records_give_the_same_bits(engine, stream_scans):
    n = 12
    s32 = [s.astype(np.float32) for s in stream_scans[:n]]
    runs = []
    for kind in ("f32x3", "f32x4", "f64"):
        odom = slam_b200.Odometry(engine)
        got = []
        for i in range(n):
            if kind == "f32x3":
                p = s32[i]
            elif kind == "f32x4":   # KITTI records: x, y, z, intensity
                p = np.concatenate([s32[i], np.full((len(s32[i]), 1), 0.25, dtype=np.float32)], axis=1)
            else:
                p = s32[i].astype(np.float64)
            got.append(frame_bits(odom.push(p, i, want_cloud=True, want_world_f32=True, want_desc=True)))
        odom.close()
        runs.append(got)
    for other in runs[1:]:
        assert all(same_bits(a, b) for a, b in zip(runs[0], other))


@pytest.mark.gpu
def test_skipped_frame_keeps_the_previous_target(engine, stream_scans):
    det = loop_detector(engine)
    odom = slam_b200.Odometry(engine, loop=det)
    frames = [odom.push(stream_scans[i], i) for i in range(5)]
    size = det.size()
    sparse = stream_scans[5][::200]          # a few dozen rows: fewer than min_points after the voxel grid
    f = odom.push(sparse, 5, detect=False, want_cloud=True)
    assert f.state == slam_b200.ODOM_SKIPPED and 0 < f.n_points < 1000
    assert same_bits(f.cloud, engine.voxel_downsample(sparse, VOXEL))
    assert same_bits(f.pose, frames[-1].pose) and f.icp is None and f.world_f32 is None
    assert det.size() == size
    nxt = odom.push(stream_scans[6], 6)
    assert nxt.state == slam_b200.ODOM_REGISTERED
    want = engine.icp_point_to_plane(engine.voxel_downsample(stream_scans[6], VOXEL),
                                     engine.voxel_downsample(stream_scans[4], VOXEL), engine.icp_config())
    assert same_bits(icp_bits(nxt.icp), icp_bits(want))
    assert det.size() == size + 1
    odom.close()
    det.close()


@pytest.mark.gpu
def test_set_pose_continues_the_chain(engine, stream_scans):
    odom = slam_b200.Odometry(engine)
    for i in range(3):
        odom.push(stream_scans[i], i)
    c, s = np.cos(0.3), np.sin(0.3)
    P = np.array([[c, -s, 0.0, 12.5], [s, c, 0.0, -3.25], [0.0, 0.0, 1.0, 0.125], [0.0, 0.0, 0.0, 1.0]])
    odom.set_pose(P)
    assert same_bits(odom.pose, P)
    f = odom.push(stream_scans[3], 3)
    r = f.icp
    keep = r.status == 0 and r.converged and not (r.final_error > 1.0)
    assert same_bits(f.pose, host_pose_product(P, r.transformation if keep else np.eye(4)))
    assert same_bits(odom.pose, f.pose)
    odom.close()


@pytest.mark.gpu
def test_add_frame_into_a_sharded_detector(engine, stream_scans):
    """world 2 (rank 0 and rank 1 objects on one context): every frame pushed with SB_ODOM_ADD_FRAME leaves each rank's
    detector as sb_loop_add_frame of the downsampled frame does (owned entries plus the newest as a guest)."""
    n = 14

    def det(rank):
        return slam_b200.LoopClosureDetector(engine, frame_gap=3, sc_distance_threshold=1e300, rank=rank, world=2)

    sess, ref = [det(0), det(1)], [det(0), det(1)]
    odoms = [slam_b200.Odometry(engine, loop=d) for d in sess]
    for i in range(n):
        clouds = [o.push(stream_scans[i], i, want_cloud=True).cloud for o in odoms]
        assert same_bits(clouds[0], clouds[1])
        for r in ref:
            r.addFrame(clouds[0], i)
        for a, b in zip(sess, ref):
            assert a.size() == b.size() == i + 1
            assert all(same_bits(x, y) for x, y in zip(a.candidates_local(), b.candidates_local())), i
    for o in odoms:
        o.close()
    for d in sess + ref:
        d.close()


@pytest.mark.gpu
def test_failed_pushes_leave_the_session_unchanged(stream_scans):
    """A NaN row (SB_ERR_RANGE), an empty frame with min_points 0 (SB_ERR_EMPTY), SB_ODOM_DETECT without a detector or
    with a world-2 one (SB_ERR_INVALID_ARG): the remaining frames give the bits of a session that never saw the bad
    calls.  In a child process (tests/odom_worker.py), so that the engine of this test session is not shared with it."""
    with tempfile.TemporaryDirectory() as d:
        for i in range(10):
            np.save(os.path.join(d, f"scan_{i}.npy"), stream_scans[i])
        p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "odom_worker.py"), d], capture_output=True,
                           text=True, timeout=900)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "ODOM_WORKER_OK" in p.stdout, p.stdout + p.stderr


@pytest.mark.gpu
def test_mirror_odometry_matches_the_single_call_api():
    with tempfile.TemporaryDirectory() as d:
        exe = build_mirror_test(d)
        p = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "all checks passed" in p.stdout
