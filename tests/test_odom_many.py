"""Many streaming sessions in one call (sb_odom_push_many, slam_b200.push_many): every output of every call, and every
session, detector and map afterwards, must be bit-identical to the same sessions driven frame by frame with
sb_odom_push in array order (test_odom_session.py pins that path to the per-call loop and the oracle).  Scans come from
the device raycaster (sb_synth_scans_dev, bit-identical to the host raycaster: test_scale_parity.py), on different
scenes and trajectories per stream, at voxel 0.5."""
import ctypes as C
import os
import random
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "lidar-slam-from-scratch_b200", "python"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import oracle_lib  # noqa: E402
import slam_b200  # noqa: E402
from test_odom_session import STREAM_FRAMES, STREAM_RADIUS, STREAM_SCENE, frame_bits, loop_bits, node_detects, same_bits  # noqa: E402,E501

VOXEL = 0.5
ALL_OUT = dict(want_cloud=True, want_world_f32=True, want_desc=True)


# ------------------------------------------------------------------ CPU
def test_push_many_of_nothing_is_a_no_op_and_null_sessions_are_refused():
    lib = slam_b200.load_library()
    assert lib.sb_odom_push_many(None, 0, None, None, None, None, None, None, None, None, None, None) == 0
    assert lib.sb_odom_push_many_f32(None, 0, None, 4, None, None, None, None, None, None, None, None, None) == 0
    assert lib.sb_odom_push_many(None, 1, None, None, None, None, None, None, None, None, None, None) == 1
    assert lib.sb_odom_push_many(None, -1, None, None, None, None, None, None, None, None, None, None) == 1
    assert slam_b200.push_many([], [], []) == []


def test_mirror_push_many_compiles():
    """slam::b200::Odometry::push_many over the mirror headers (compile only)."""
    import subprocess
    import tempfile
    prog = r'''
#include "slam_viz/core/odometry.hpp"
std::vector<slam::b200::OdometryFrame> f(std::vector<slam::b200::Odometry*>& s, std::vector<slam::PointCloud>& c) {
  return slam::b200::Odometry::push_many(s, c, std::vector<int>(s.size(), 0), true, false, true);
}
'''
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "t.cpp")
        with open(src, "w") as fh:
            fh.write(prog)
        subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Wno-unused-function", "-fsyntax-only",
                               "-I" + os.path.join(ROOT, "include"),
                               "-I" + os.path.join(ROOT, "lidar-slam-from-scratch_b200", "host"), src])


# ------------------------------------------------------------------ helpers
def device_scans(engine, sensor, world, poses, seed):
    """Scans at `poses` (n, 3) from the device raycaster, as host fp64 arrays."""
    import torch
    rays = sensor["beams"] * sensor["azimuth_steps"]
    d = torch.empty(len(poses) * rays * 3, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    off = engine.synth_scans_dev(sensor, world, np.asarray(poses, dtype=np.float64), seed, d.data_ptr())
    engine.synchronize()
    h = d[:int(off[-1]) * 3].cpu().numpy().reshape(-1, 3)
    return [h[off[i]:off[i + 1]].copy() for i in range(len(poses))]


_STREAMS = {}


def streams(engine, synth, n, frames=12, sensor=None):
    """n streams of `frames` scans, each on its own scene (8 scenes, re-used with other trajectories beyond 8)."""
    sensor = sensor or oracle_lib.SENSOR64
    key = (n, frames, sensor["beams"], sensor["azimuth_steps"])
    if key not in _STREAMS:
        out = []
        for s in range(n):
            world = synth.scene(40 + s % 8, n_boxes=400)
            start, lateral = 3.0 * (s // 8), 0.7 * ((s % 3) - 1)
            poses = [synth.pose(0, 0.0, start + 0.9 * i, lateral) for i in range(frames)]
            out.append(device_scans(engine, sensor, world, poses, 9000 + 131 * s))
        _STREAMS[key] = out
    return _STREAMS[key]


def loop_detector(engine):
    return slam_b200.LoopClosureDetector(engine, frame_gap=50, sc_distance_threshold=0.25, icp_fitness_threshold=0.3,
                                         max_candidates=3)


def sessions(engine, n, loop=False, map=False, **kw):
    return [slam_b200.Odometry(engine, voxel=VOXEL, loop=loop_detector(engine) if loop else None,
                               map=slam_b200.Map(engine) if map else None, **kw) for _ in range(n)]


def close(objs):
    for o in objs:
        for x in (o, o.loop, o.map):
            if x is not None:
                x.close()


def assert_same(got, want, what):
    assert len(got) == len(want), what
    for j, (a, b) in enumerate(zip(got, want)):
        assert same_bits(frame_bits(a), frame_bits(b)), (what, j, a.state, b.state)


def kernel_names(fn):
    """Names of the kernels fn launches (torch.profiler with CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


# ------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 8, 64])
def test_equal_to_single_pushes_across_n(engine, synth, n):
    data = streams(engine, synth, n)
    ref, many = sessions(engine, n), sessions(engine, n)
    names = None
    for i in range(len(data[0])):
        want = [o.push(data[s][i], i, **ALL_OUT) for s, o in enumerate(ref)]
        call = lambda: slam_b200.push_many(many, [d[i] for d in data], i, **ALL_OUT)  # noqa: E731
        if i == 3:   # which normals path the batch took: the small-batch k_knn<1> or the packet k_self_knn + redo
            out = []
            names = kernel_names(lambda: out.append(call()))
            got = out[0]
        else:
            got = call()
        assert_same(got, want, (n, i))
        assert all(f.state == (slam_b200.ODOM_FIRST if i == 0 else slam_b200.ODOM_REGISTERED) for f in got)
    for a, b in zip(ref, many):
        assert same_bits(a.pose, b.pose)
    packet = any("k_self_knn" in x for x in names)
    small = any("k_knn<1>" in x for x in names)
    assert packet != small, sorted(names)
    # forest.cu: the packet path once the batch gives every SM >= 24 warps of 32 queries (148 SMs: ~15 scans of ~8 k rows)
    assert packet == (n >= 64) and small == (n <= 8), (n, sorted(x for x in names if "knn" in x))
    if packet:
        assert any("k_knn_redo" in x for x in names) and any("k_normals_from_graph" in x for x in names)
    print(f"[odom_many] n={n}: {len(data[0])} calls bit-identical to single pushes, normals path "
          f"{'packet' if packet else 'small-batch'}")
    close(ref + many)


@pytest.fixture(scope="module")
def loop_streams(engine, synth):
    import bench
    world = synth.scene(STREAM_SCENE, n_boxes=400, path_kind=1, radius=STREAM_RADIUS)
    poses = [synth.pose(1, STREAM_RADIUS, float(i)) for i in range(STREAM_FRAMES)]
    return [device_scans(engine, bench.SENSOR, world, poses, 500 + 1000 * s) for s in range(4)]


@pytest.mark.gpu
def test_loop_closure_and_map(engine, loop_streams):
    ref, many = sessions(engine, 4, loop=True, map=True), sessions(engine, 4, loop=True, map=True)
    accepted = 0
    for i in range(STREAM_FRAMES):
        kw = dict(add_frame=True, detect=node_detects(i), add_map=True, want_cloud=True, want_world_f32=True)
        want = [o.push(loop_streams[s][i], i, **kw) for s, o in enumerate(ref)]
        got = slam_b200.push_many(many, [d[i] for d in loop_streams], i, **kw)
        assert_same(got, want, i)
        for f, w in zip(got, want):
            assert [loop_bits(x).tolist() for x in f.loops] == [loop_bits(x).tolist() for x in w.loops]
            accepted += len(f.loops)
    for a, b in zip(ref, many):
        assert a.loop.size() == b.loop.size() == STREAM_FRAMES
        assert all(same_bits(x, y) for x, y in zip(a.loop.candidates_local(), b.loop.candidates_local()))
        ca, cb = a.map.occupancy_cells(), b.map.occupancy_cells()
        assert ca[1] == cb[1] and np.array_equal(ca[0], cb[0])
        assert same_bits(a.map.global_map(2 * VOXEL), b.map.global_map(2 * VOXEL))
        assert same_bits(a.map.poses(), b.map.poses())
    assert accepted >= 4, "every stream revisits its start: detect() must accept loop closures"
    print(f"[odom_many] 4 streams x {STREAM_FRAMES} frames with detector and map: identical, {accepted} loops")
    close(ref + many)


@pytest.mark.gpu
def test_sessions_at_different_stages(engine, synth):
    data = streams(engine, synth, 8)
    c, s = np.cos(0.4), np.sin(0.4)
    P0 = np.array([[c, -s, 0.0, 5.5], [s, c, 0.0, -2.0], [0.0, 0.0, 1.0, 0.25], [0.0, 0.0, 0.0, 1.0]])
    kws = [dict(), dict(), dict(min_points=10 ** 6), dict(max_error=0.02, initial_pose=P0), dict(max_error=1e-12)]
    ref = [slam_b200.Odometry(engine, voxel=VOXEL, **kw) for kw in kws]
    many = [slam_b200.Odometry(engine, voxel=VOXEL, **kw) for kw in kws]
    for o, m in zip(ref[1:], many[1:]):   # all but session 0 have seen a frame
        o.push(data[1][0], 0)
        m.push(data[1][0], 0)
    for step in range(4):
        frames = [data[s][step + 1] for s in range(len(kws))]
        want = [o.push(f, step + 1, **ALL_OUT) for o, f in zip(ref, frames)]
        got = slam_b200.push_many(many, frames, step + 1, **ALL_OUT)
        assert_same(got, want, step)
        if step == 0:
            assert [f.state for f in got] == [slam_b200.ODOM_FIRST, slam_b200.ODOM_REGISTERED, slam_b200.ODOM_SKIPPED,
                                              slam_b200.ODOM_REGISTERED, slam_b200.ODOM_REGISTERED]
    close(ref + many)


@pytest.mark.gpu
def test_mixing_single_and_many_pushes_and_subsets(engine, synth):
    data = streams(engine, synth, 8)
    n = 5
    ref, many = sessions(engine, n, loop=True), sessions(engine, n, loop=True)
    nxt = [0] * n
    rng = random.Random(7)
    for call in range(10):
        if call % 2:
            s = rng.randrange(n)
            want = [ref[s].push(data[s][nxt[s]], nxt[s], **ALL_OUT)]
            got = [many[s].push(data[s][nxt[s]], nxt[s], **ALL_OUT)]
            nxt[s] += 1
        else:
            sub = rng.sample(range(n), rng.randint(2, n))
            want = [ref[s].push(data[s][nxt[s]], nxt[s], **ALL_OUT) for s in sub]
            got = slam_b200.push_many([many[s] for s in sub], [data[s][nxt[s]] for s in sub], [nxt[s] for s in sub], **ALL_OUT)
            for s in sub:
                nxt[s] += 1
        assert_same(got, want, call)
    for a, b in zip(ref, many):
        assert a.loop.size() == b.loop.size()
        assert all(same_bits(x, y) for x, y in zip(a.loop.candidates_local(), b.loop.candidates_local()))
    close(ref + many)


@pytest.mark.gpu
@pytest.mark.parametrize("reserve", [False, True])
def test_growing_and_shrinking_frames(engine, synth, reserve):
    sensors = [oracle_lib.small_sensor(16, 300), oracle_lib.SENSOR64, oracle_lib.small_sensor(32, 600),
               oracle_lib.SENSOR128, oracle_lib.small_sensor(16, 300), oracle_lib.SENSOR128]
    n = 3
    data = [[streams(engine, synth, n, frames=len(sensors), sensor=sen)[s][k] for k, sen in enumerate(sensors)]
            for s in range(n)]
    for f32 in (False, True):
        ref, many = sessions(engine, n, min_points=200), sessions(engine, n, min_points=200)
        if reserve:
            for o in ref + many:
                o.reserve(max(len(x) for d in data for x in d) // 2)   # too small for the largest frames
        for k in range(len(sensors)):
            def rows(s):
                x = data[s][k]
                if not f32:
                    return x
                return np.concatenate([x.astype(np.float32), np.full((len(x), 1), 0.5, dtype=np.float32)], axis=1)
            want = [o.push(rows(s), k, **ALL_OUT) for s, o in enumerate(ref)]
            got = slam_b200.push_many(many, [rows(s) for s in range(n)], k, **ALL_OUT)
            assert_same(got, want, (f32, k))
        close(ref + many)


def _check_fails(fn, status, text=None):
    with pytest.raises(slam_b200.SlamB200Error) as e:
        fn()
    assert e.value.status == status, str(e.value)
    if text is not None:
        assert text in str(e.value), str(e.value)


@pytest.mark.gpu
def test_failure_is_atomic(engine, synth):
    data = streams(engine, synth, 8)
    n = 4
    ref, many = sessions(engine, n, loop=True, map=True), sessions(engine, n, loop=True, map=True)
    kw = dict(ALL_OUT, add_frame=True, add_map=True)
    for i in range(3):
        assert_same(slam_b200.push_many(many, [d[i] for d in data[:n]], i, **kw),
                    [o.push(data[s][i], i, **kw) for s, o in enumerate(ref)], i)
    bad = [d[3].copy() for d in data[:n]]
    bad[2][17, 1] = np.nan
    _check_fails(lambda: slam_b200.push_many(many, bad, 3, **kw), 5, "session 2")
    empty = [d[3] for d in data[:n]]
    empty[1] = np.zeros((0, 3))
    zero = sessions(engine, n, min_points=0)
    _check_fails(lambda: slam_b200.push_many(zero, empty, 0), 2, "session 1")   # SB_ERR_EMPTY
    close(zero)
    for i in range(3, 6):
        want = [o.push(data[s][i], i, **kw) for s, o in enumerate(ref)]
        got = slam_b200.push_many(many, [d[i] for d in data[:n]], i, **kw)
        assert_same(got, want, i)
    for a, b in zip(ref, many):
        assert a.loop.size() == b.loop.size() and len(a.map) == len(b.map)
        assert all(same_bits(x, y) for x, y in zip(a.loop.candidates_local(), b.loop.candidates_local()))
        assert np.array_equal(a.map.occupancy_cells()[0], b.map.occupancy_cells()[0])
        assert same_bits(a.map.global_map(0.0), b.map.global_map(0.0))
    close(ref + many)


@pytest.mark.gpu
def test_argument_rules(engine, synth):
    import torch
    data = streams(engine, synth, 8)
    ref, many = sessions(engine, 3), sessions(engine, 3)
    f0 = [d[0] for d in data[:3]]
    want = [o.push(f, 0, **ALL_OUT) for o, f in zip(ref, f0)]
    assert_same(slam_b200.push_many(many, f0, 0, **ALL_OUT), want, 0)
    f1 = [d[1] for d in data[:3]]
    e2 = slam_b200.Engine(0)
    other = slam_b200.Odometry(e2, voxel=VOXEL)
    det = loop_detector(engine)
    mp = slam_b200.Map(engine)
    shared_det = [slam_b200.Odometry(engine, voxel=VOXEL, loop=det) for _ in range(2)]
    shared_map = [slam_b200.Odometry(engine, voxel=VOXEL, map=mp) for _ in range(2)]
    sharded = slam_b200.LoopClosureDetector(engine, rank=0, world=2)
    with_sharded = slam_b200.Odometry(engine, voxel=VOXEL, loop=sharded)
    cfg = engine.icp_config(max_iterations=30)
    bad_cfg = slam_b200.Odometry(engine, voxel=VOXEL, cfg=cfg)
    bad_voxel = slam_b200.Odometry(engine, voxel=0.4)
    dev = torch.from_numpy(f1[1]).cuda()
    cases = [
        ("appears twice", [many[0], many[1], many[0]], f1),
        ("another context", [many[0], other], f1[:2]),
        ("shares its loop-closure detector", shared_det, f1[:2]),
        ("shares its map", shared_map, f1[:2]),
        ("another voxel or icp config", [many[0], bad_cfg], f1[:2]),
        ("another voxel or icp config", [many[0], bad_voxel], f1[:2]),
        ("world == 1", [many[0], with_sharded], f1[:2]),
    ]
    for text, ss, fr in cases:
        _check_fails(lambda: slam_b200.push_many(ss, fr, 1, detect=(text == "world == 1")), 1, text)
    # a device pointer as rows, through the C ABI
    lib = engine.lib
    hs = (C.c_void_p * 2)(many[0].h, many[1].h)
    xs = (C.c_void_p * 2)(f1[0].ctypes.data, dev.data_ptr())
    rows = np.array([len(f1[0]), len(f1[1])], dtype=np.int64)
    fi = np.array([1, 1], dtype=np.int32)
    out = (slam_b200.OdomFrameC * 2)()
    s = lib.sb_odom_push_many(hs, 2, xs, rows.ctypes.data_as(slam_b200._I64), fi.ctypes.data_as(slam_b200._I32), None,
                              out, None, None, None, None, None)
    assert s == 1 and b"session 1" in lib.sb_last_error(engine.h)
    torch.cuda.synchronize()
    # nothing changed: the next calls give the bits of sessions that never saw the refused ones
    for i in (1, 2):
        want = [o.push(d[i], i, **ALL_OUT) for o, d in zip(ref, data[:3])]
        assert_same(slam_b200.push_many(many, [d[i] for d in data[:3]], i, **ALL_OUT), want, i)
    close(ref + many + shared_det + shared_map + [with_sharded, bad_cfg, bad_voxel])
    other.close()
    e2.close()


@pytest.mark.gpu
def test_launches_do_not_grow_with_n(engine, synth):
    data = streams(engine, synth, 64)
    per = {}
    for n in (8, 64):
        many = sessions(engine, n)
        slam_b200.push_many(many, [d[0] for d in data[:n]], 0)
        counts, iters = [], []
        for i in range(1, 6):
            l0 = engine.launch_count
            got = slam_b200.push_many(many, [d[i] for d in data[:n]], i)
            counts.append(engine.launch_count - l0)
            iters.append(max(f.icp.num_iterations for f in got))
        per[n] = (counts, iters)
        close(many)
    single = sessions(engine, 64)
    for s, o in enumerate(single):
        o.push(data[s][0], 0)
    l0 = engine.launch_count
    for s, o in enumerate(single):
        o.push(data[s][1], 1)
    singles = engine.launch_count - l0
    close(single)
    # the ICP loop's launches grow with the batch's longest pair (4 per pass); everything else is per call
    base = {n: [c - 4 * it for c, it in zip(*per[n])] for n in per}
    assert max(base[64]) - min(base[8]) <= 4 and max(base[8]) - min(base[64]) <= 4, per
    assert per[64][0][0] < singles, (per, singles)
    print(f"[odom_many] launches per call: n=8 {per[8][0]}, n=64 {per[64][0]} (longest ICP {per[8][1]}, {per[64][1]}); "
          f"64 single pushes {singles}")
