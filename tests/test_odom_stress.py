"""The streaming odometry session (sb_odom_*, csrc/odom.cu) on the streams test_odom_session.py does not send: frames
that grow and shrink so that both ping-pong slots regrow while the other one holds the ICP target, frames above the
one-CTA sort capacity, fp64 rows that take the voxel grid's sort path, pinned input, every configuration field, every
output subset, other work on the same context between pushes, and what the node publishes from the session's poses.

Each stream is checked bit for bit against the node's per-call loop over the single-call API (voxel_downsample,
icp_point_to_plane, odometry_poses, transform_clouds_f32, sc_compute, addFrame / detect_batch), and against the
oracle where the per-call loop has not been checked at that shape.
"""
import ctypes as C
import os
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "lidar-slam-from-scratch_b200", "python"))
import bench  # noqa: E402
import oracle_lib  # noqa: E402
import slam_b200  # noqa: E402
from test_odom_session import STREAM_RADIUS, STREAM_SCENE, VOXEL, frame_bits, icp_bits, loop_bits, same_bits  # noqa: E402
from test_scale_parity import compare_icp, margin, node_delta, rot_angle  # noqa: E402

WORKER = os.path.join(HERE, "odom_stress_worker.py")
SEG_CAP = 12288          # scan_sort.cu: longest segment the one-CTA shared-memory sort takes
SC_BYTES = slam_b200.SB_SC_SIZE * 8
ALL = dict(want_cloud=True, want_world_f32=True, want_desc=True)


def cores():
    return os.cpu_count() or 1


# ------------------------------------------------------------------ the per-call loop
def icp_batch(r):
    """One ICPResult as the one-record batch sb_odometry_poses takes."""
    rec = np.zeros(1, dtype=slam_b200.ICP_DTYPE)
    rec[0]["transformation"] = r.transformation.reshape(16)
    rec[0]["final_error"], rec[0]["converged"], rec[0]["num_iterations"] = r.final_error, r.converged, r.num_iterations
    rec[0]["status"], rec[0]["history_len"] = r.status, len(r.error_history)
    rec[0]["error_history"][:len(r.error_history)] = r.error_history
    return slam_b200.ICPResultBatch(rec)


def per_call_loop(engine, scans, voxel=VOXEL, cfg=None, max_error=1.0, min_points=1000, initial_pose=None, det=None,
                  detect=()):
    """SlamNode::process_frame over the single-call entry points: per frame a dict with what an OdomFrame carries when
    every output is asked for.  A frame with fewer than min_points rows is skipped (pose repeated, target kept).
    det: a detector that gets addFrame of every kept frame; detect: frame indices whose detect_batch is recorded."""
    cfg = cfg or engine.icp_config()
    pose = np.eye(4) if initial_pose is None else np.array(initial_pose, dtype=np.float64).reshape(4, 4)
    prev, out = None, []
    for i, scan in enumerate(scans):
        cur = engine.voxel_downsample(scan, voxel)
        f = dict(frame_idx=i, n_points=len(cur), cloud=cur, icp=None, world=None, desc=None, loops=[])
        if len(cur) < min_points:
            f.update(state=slam_b200.ODOM_SKIPPED, pose=pose.copy())
            out.append(f)
            continue
        if prev is None:
            f["state"] = slam_b200.ODOM_FIRST
        else:
            f["state"] = slam_b200.ODOM_REGISTERED
            f["icp"] = engine.icp_point_to_plane(cur, prev, cfg)
            pose = engine.odometry_poses(icp_batch(f["icp"]), max_error=max_error, initial_pose=pose)[1]
        f["pose"] = pose.copy()
        f["world"] = engine.transform_clouds_f32(cur, np.array([0, len(cur)], dtype=np.int64), pose[None])
        f["desc"] = engine.sc_compute(cur)
        if det is not None:
            det.addFrame(cur, i)
            if i in detect:
                f["loops"] = det.detect_batch([det.size() - 1])[0]
        prev = cur
        out.append(f)
    return out


def want_bits(f):
    """frame_bits of the OdomFrame the session should return for per_call_loop's frame f, every output asked for."""
    parts = [[f["frame_idx"], f["state"], f["n_points"], len(f["loops"])], f["pose"].reshape(16),
             icp_bits(f["icp"]) if f["icp"] is not None else [], f["cloud"].reshape(-1),
             [] if f["world"] is None else f["world"].astype(np.float64).reshape(-1),
             [] if f["desc"] is None else f["desc"]]
    parts += [loop_bits(r) for r in f["loops"]]
    return np.concatenate([np.asarray(p, dtype=np.float64).reshape(-1) for p in parts])


def run_session(engine, scans, loop=None, detect=(), reserve=None, **kw):
    odom = slam_b200.Odometry(engine, loop=loop, **kw)
    if reserve is not None:
        odom.reserve(reserve)
    frames = [odom.push(s, i, detect=i in detect, **ALL) for i, s in enumerate(scans)]
    odom.close()
    return frames


def assert_matches_per_call(frames, want, what):
    assert len(frames) == len(want)
    for i, (f, w) in enumerate(zip(frames, want)):
        assert f.state == w["state"] and f.n_points == w["n_points"], (what, i, f.state, f.n_points, w["n_points"])
        assert same_bits(frame_bits(f), want_bits(w)), (what, i)


# ------------------------------------------------------------------ slot growth: a model of odom.cu's allocations
OUT_ROWS = 16 * 8 + SC_BYTES


def _grow(cap, need):
    """grow_dev / grow_host: the new capacity and whether it grew."""
    if need <= cap:
        return cap, False
    c = cap if cap > 0 else need
    while c < need:
        c *= 2
    return c, True


def _tree_need(n):
    """tree_store_need (forest.cu): boxes and seed-grid slots of one tree of n points."""
    nb, cnt = 0, (n + 31) // 32
    while True:
        nb += cnt
        if cnt <= 32:
            break
        cnt = (cnt + 31) // 32
    lg = 6
    while (1 << lg) < 2 * n:
        lg += 1
    return nb, 1 << lg


def growth_events(raw_rows, kept_rows, min_points, row_bytes=24, pinned=False):
    """Replays push_impl's buffer growth (slot_reserve, out_reserve, d_raw, h_in) for a stream of frames with raw_rows
    input rows and kept_rows rows after the voxel grid.  Returns (frame, site, slot, other slot holds the target)."""
    slots = [dict(xyz=0, points=0, grid=0, boxes=0) for _ in range(2)]
    shared = dict(d_raw=0, h_in=0, d_out=0)
    prev, events = -1, []

    def reserve(i, s, raw, pts):
        S = slots[s]
        for site, need in (("xyz", 3 * max(raw, 1)), ("points", pts), ("grid", _tree_need(max(pts, 1))[1]),
                           ("boxes", _tree_need(max(pts, 1))[0])):
            S[site], grew = _grow(S[site], need)
            if grew:
                events.append((i, site, s, prev >= 0))

    def shared_grow(i, site, need):
        shared[site], grew = _grow(shared[site], need)
        if grew:
            events.append((i, site, None, prev >= 0))

    for i, (n, m) in enumerate(zip(raw_rows, kept_rows)):
        s = 0 if prev < 0 else 1 - prev
        reserve(i, s, n, 0)
        shared_grow(i, "d_raw", max(n * row_bytes, 1))
        if n > 0 and not pinned:
            shared_grow(i, "h_in", n * row_bytes)
        if m < min_points:
            continue
        reserve(i, s, n, m)
        shared_grow(i, "d_out", OUT_ROWS + 36 * max(m, 1))
        prev = s
    return events


# ------------------------------------------------------------------ CPU
def test_growth_model_matches_the_allocator():
    """The model of the growth test: doubling from the first need, the four per-point arrays as one site."""
    assert _grow(0, 10) == (10, True) and _grow(10, 10) == (10, False) and _grow(10, 11) == (20, True)
    assert _grow(10, 41) == (80, True)
    assert _tree_need(1) == (1, 64) and _tree_need(33) == (2, 128) and _tree_need(2048) == (66, 4096)
    ev = growth_events([100, 100, 5000, 10, 6000], [1000, 1000, 3000, 5, 4000], 1000)
    assert ("points", 0) in [(e[1], e[2]) for e in ev if e[0] == 2 and e[3]]   # frame 2: slot 0, slot 1 holds target
    assert not [e for e in ev if e[0] == 3 and e[1] in ("points", "d_out")]     # skipped frame: no tree, no outputs
    assert ("points", 1) in [(e[1], e[2]) for e in ev if e[0] == 4 and e[3]]   # frame 4: slot 1 (the skip kept slot 0)


def test_handles_outliving_their_engine_do_not_touch_its_context():
    """A session, detector or index closed (or collected) after Engine.close() -- e.g. one a failing test left open --
    drops its handle: the context its free would use is gone."""
    class Lib:
        def __getattr__(self, name):
            raise AssertionError(f"{name} called after the engine was closed")

    class ClosedEngine:
        h, lib = None, Lib()

    for cls in (slam_b200.Odometry, slam_b200.LoopClosureDetector, slam_b200.KDTree):
        obj = cls.__new__(cls)
        obj.e, obj.h = ClosedEngine(), C.c_void_p(1)
        obj.close()
        assert obj.h is None, cls


def test_worker_argument_handling():
    """The child process of the forced-path test refuses to run without its directory or without its switches."""
    env = {k: v for k, v in os.environ.items() if k not in ("SB_SORT_TILED", "SB_VOXEL_SORT")}
    p = subprocess.run([sys.executable, WORKER], capture_output=True, text=True, timeout=120, env=env)
    assert p.returncode == 2 and "usage" in p.stderr, p.stdout + p.stderr
    with tempfile.TemporaryDirectory() as d:
        p = subprocess.run([sys.executable, WORKER, d], capture_output=True, text=True, timeout=120, env=env)
        assert p.returncode == 2 and "SB_SORT_TILED=1 SB_VOXEL_SORT=1" in p.stderr, p.stdout + p.stderr
        env.update(SB_SORT_TILED="1", SB_VOXEL_SORT="1")
        p = subprocess.run([sys.executable, WORKER, os.path.join(d, "missing")], capture_output=True, text=True,
                           timeout=120, env=env)
        assert p.returncode == 2 and "no frames" in p.stderr, p.stdout + p.stderr


# ------------------------------------------------------------------ GPU fixtures
@pytest.fixture(scope="module")
def stream(synth):
    """The first 40 frames of test_odom_session's loop-closure sequence (bench.SENSOR, noise seeds 500 + i)."""
    world = synth.scene(STREAM_SCENE, n_boxes=400, path_kind=1, radius=STREAM_RADIUS)
    return [synth.scan(bench.SENSOR, world, synth.pose(1, STREAM_RADIUS, float(i)), 500 + i, threads=cores())
            for i in range(40)]


GROW_KINDS = ["s16", "s16", "s32", "s32", "s16", "s16", "s16", "bench", "skip", "bench", "bench", "s32", "s16", "s32",
              "bench", "bench"]


@pytest.fixture(scope="module")
def growing_stream(synth, scene):
    """16 frames a metre apart in one scene from three sensors: small -> large -> small -> larger, with a frame below
    min_points between two growth steps."""
    sensors = dict(s16=oracle_lib.small_sensor(16, 360), s32=oracle_lib.small_sensor(32, 600), bench=bench.SENSOR)
    out = []
    for i, kind in enumerate(GROW_KINDS):
        s = sensors["bench" if kind == "skip" else kind]
        scan = synth.scan(s, scene, (float(i), 0.0, 0.0), 600 + i, threads=cores())
        out.append(scan[::200].copy() if kind == "skip" else scan)
    return out


def pinned(rows, dtype):
    import torch
    t = torch.empty(rows.shape, dtype=dtype, pin_memory=True)
    a = t.numpy()
    a[...] = rows
    assert t.is_pinned() and a.ctypes.data == t.data_ptr()
    return t, a


# ------------------------------------------------------------------ 1. growing stream, no reserve
@pytest.mark.gpu
def test_growing_stream_regrows_both_slots_with_the_per_call_bits(engine, growing_stream):
    scans = growing_stream
    want = per_call_loop(engine, scans)
    frames = run_session(engine, scans)
    assert_matches_per_call(frames, want, "growing")
    kept = [f.n_points for f in frames]
    assert [f.state == slam_b200.ODOM_SKIPPED for f in frames] == [k == "skip" for k in GROW_KINDS]
    ev = growth_events([len(s) for s in scans], kept, 1000)
    mid = [e for e in ev if e[3]]     # the other slot holds the previous frame, the ICP target of this one
    counts = {}
    for _, site, slot, _ in mid:
        counts[(site, slot)] = counts.get((site, slot), 0) + 1
    for site in ("xyz", "points", "grid", "boxes"):
        for slot in (0, 1):
            assert counts.get((site, slot), 0) >= 1, (site, slot, ev)
    for site in ("d_raw", "h_in", "d_out"):
        assert counts.get((site, None), 0) >= 1, (site, ev)
    # the skipped frame sits between two growth steps of the per-point arrays
    skip = GROW_KINDS.index("skip")
    grew = sorted({e[0] for e in mid if e[1] == "points"})
    assert any(g < skip for g in grew) and any(g > skip for g in grew), grew
    print(f"[odom-stress] growing stream: raw {[len(s) for s in scans]}, kept {kept}; buffers grown while the other "
          f"slot held the target: " + ", ".join(f"{site}{'' if slot is None else '@' + str(slot)}={c}"
                                               for (site, slot), c in sorted(counts.items(), key=str)))
    # reserve(): too small (every buffer still grows on demand), then ample (nothing grows): the same bits
    ref = [frame_bits(f) for f in frames]
    for size in (1000, max(len(s) for s in scans)):
        again = run_session(engine, scans, reserve=size)
        assert all(same_bits(frame_bits(f), r) for f, r in zip(again, ref)), size


# ------------------------------------------------------------------ 2. large frames across the sort capacity
@pytest.mark.gpu
def test_large_frames_above_the_sort_capacity_match_per_call_and_oracle(engine, oracle, stream):
    voxel, n = 0.2, 8
    scans = stream[:n]
    want = per_call_loop(engine, scans, voxel=voxel)
    frames = run_session(engine, scans, voxel=voxel)
    assert_matches_per_call(frames, want, "voxel 0.2")
    sizes = [f.n_points for f in frames]
    assert min(sizes) > SEG_CAP, sizes
    ocl = [oracle.voxel_downsample(s, voxel)[0] for s in scans]
    for f, o in zip(frames, ocl):
        assert same_bits(f.cloud, o)
    with ThreadPoolExecutor(cores()) as ex:
        oicp = [None] + list(ex.map(lambda i: oracle.icp_point_to_plane(ocl[i], ocl[i - 1]), range(1, n)))
    assert min(margin(o["error_history"]) for o in oicp[1:]) > 1e-12
    P, worst = np.eye(4), (0.0, 0.0)
    for i in range(1, n):
        dt, dr = compare_icp(frames[i].icp, oicp[i])
        worst = (max(worst[0], dt), max(worst[1], dr))
        o = oicp[i]
        P = P @ node_delta(o["converged"], o["final_error"], o["transformation"])
        dP = frames[i].pose @ np.linalg.inv(P)
        assert np.linalg.norm(dP[:3, 3]) < 1e-4 and rot_angle(dP[:3, :3]) < 1e-5, i
    print(f"[odom-stress] voxel {voxel}: {sizes} rows per frame (sort capacity {SEG_CAP}), worst ICP pose difference "
          f"to the oracle {worst[0]:.2e} m / {worst[1]:.2e} rad")


# ------------------------------------------------------------------ 3. forced sort paths, fp64 rows on the sort path
def jittered(scans):
    """fp64 rows that are not float32-born: the voxel grid's hashed path declines them."""
    rng = np.random.default_rng(7)
    return [s + 1e-9 * rng.standard_normal(s.shape) for s in scans]


@pytest.mark.gpu
def test_fp64_rows_take_the_voxel_sort_path_in_the_session(engine, stream):
    scans = stream[:6]
    odom = slam_b200.Odometry(engine)
    odom.push(scans[0], 0)
    assert engine.last_voxel_path == 1        # float32-born rows: hashed
    odom.close()
    rows = jittered(scans)
    want = per_call_loop(engine, rows)
    odom = slam_b200.Odometry(engine)
    frames = []
    for i, r in enumerate(rows):
        frames.append(odom.push(r, i, **ALL))
        assert engine.last_voxel_path == 2, i
    odom.close()
    assert_matches_per_call(frames, want, "fp64 jitter")
    print("[odom-stress] fp64 rows: voxel path 2 on every push")


@pytest.mark.gpu
def test_forced_tiled_and_voxel_sort_paths_reproduce_the_session(engine, stream):
    """SB_SORT_TILED and SB_VOXEL_SORT are read once per process: a child process (tests/odom_stress_worker.py) pushes
    the frames with both forced and must reproduce this process's bits."""
    scans = stream[:10]
    with tempfile.TemporaryDirectory() as d:
        for name, rows in (("plain", scans), ("jitter", jittered(scans))):
            for i, s in enumerate(rows):
                np.save(os.path.join(d, f"{name}_scan_{i}.npy"), s)
            for i, f in enumerate(run_session(engine, rows)):
                np.save(os.path.join(d, f"{name}_bits_{i}.npy"), frame_bits(f))
        env = dict(os.environ, SB_SORT_TILED="1", SB_VOXEL_SORT="1")
        p = subprocess.run([sys.executable, WORKER, d], capture_output=True, text=True, timeout=900, env=env)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "ODOM_STRESS_WORKER_OK" in p.stdout, p.stdout + p.stderr
    print("[odom-stress] " + " | ".join(line for line in p.stdout.splitlines() if line))


# ------------------------------------------------------------------ 4. input kinds
@pytest.mark.gpu
def test_pinned_and_pageable_inputs_give_the_same_bits(engine, stream):
    n = 8
    scans = stream[:n]
    s32 = [s.astype(np.float32) for s in scans]
    w64 = [s.astype(np.float64) for s in s32]
    keep = []

    def run(rows):
        odom = slam_b200.Odometry(engine)
        got = [frame_bits(odom.push(r, i, **ALL)) for i, r in enumerate(rows)]
        odom.close()
        return got

    import torch
    p64 = []
    for s in scans:
        t, a = pinned(s, torch.float64)
        assert slam_b200._f64(a, 3).ctypes.data == a.ctypes.data   # the binding passes the pinned rows through
        keep.append(t)
        p64.append(a)
    ref = run(scans)
    assert all(same_bits(a, b) for a, b in zip(run(p64), ref))
    ref32 = run(w64)
    for stride in (3, 4):
        rows = []
        for s in s32:
            r = s if stride == 3 else np.concatenate([s, np.full((len(s), 1), 0.25, dtype=np.float32)], axis=1)
            t, a = pinned(r, torch.float32)
            assert np.ascontiguousarray(a).ctypes.data == a.ctypes.data
            keep.append(t)
            rows.append(a)
        assert all(same_bits(a, b) for a, b in zip(run(rows), ref32)), stride
    # one pinned buffer, refilled for every frame and overwritten as soon as the push returns
    t, buf = pinned(np.zeros((max(len(s) for s in scans), 3)), torch.float64)
    odom = slam_b200.Odometry(engine)
    got = []
    for i, s in enumerate(scans):
        view = buf[:len(s)]
        view[...] = s
        got.append(frame_bits(odom.push(view, i, **ALL)))
        buf[...] = np.nan
    odom.close()
    assert all(same_bits(a, b) for a, b in zip(got, ref))
    print("[odom-stress] pageable fp64, pinned fp64, pinned float32 x3 / x4, reused pinned buffer: same bits")


@pytest.mark.gpu
def test_device_pointer_push_is_refused_and_leaves_the_session_unchanged(engine, stream):
    import torch
    scans = stream[:5]
    ref = [frame_bits(f) for f in run_session(engine, scans)]
    odom = slam_b200.Odometry(engine)
    got = [frame_bits(odom.push(scans[i], i, **ALL)) for i in range(3)]
    d = torch.from_numpy(scans[3]).cuda()
    torch.cuda.synchronize()
    fr = slam_b200.OdomFrameC()
    s = engine.lib.sb_odom_push(odom.h, C.cast(C.c_void_p(d.data_ptr()), C.POINTER(C.c_double)), len(scans[3]), 3, 0,
                                C.byref(fr), None, None, None, None, 0)
    assert s == 1, s                                  # SB_ERR_INVALID_ARG
    assert b"device pointer" in engine.lib.sb_last_error(engine.h)
    del d
    got += [frame_bits(odom.push(scans[i], i, **ALL)) for i in range(3, 5)]
    odom.close()
    assert all(same_bits(a, b) for a, b in zip(got, ref))


# ------------------------------------------------------------------ 5. configurations
def _config_cases(engine):
    c, s = np.cos(0.02), np.sin(0.02)
    T0 = np.array([[c, -s, 0.0, 0.3], [s, c, 0.0, 0.05], [0.0, 0.0, 1.0, 0.01], [0.0, 0.0, 0.0, 1.0]])
    P0 = np.array([[0.0, -1.0, 0.0, 4.5], [1.0, 0.0, 0.0, -2.25], [0.0, 0.0, 1.0, 0.5], [0.0, 0.0, 0.0, 1.0]])
    return [("normals_k=10", dict(cfg=engine.icp_config(normals_k=10))),
            ("normals_k=32", dict(cfg=engine.icp_config(normals_k=slam_b200.SB_MAX_K))),
            ("max_iterations=0", dict(cfg=engine.icp_config(max_iterations=0))),
            ("max_iterations=1", dict(cfg=engine.icp_config(max_iterations=1))),
            ("initial_transform", dict(cfg=engine.icp_config(initial_transform=T0))),
            ("max_error=1e-12", dict(max_error=1e-12, initial_pose=P0)),
            ("voxel=0", dict(voxel=0.0)),
            ("min_points=0", dict(min_points=0))]


@pytest.mark.gpu
def test_configurations_match_the_per_call_loop(engine, synth, stream):
    assert slam_b200.SB_MAX_K == 32
    n = 8
    world = synth.scene(STREAM_SCENE, n_boxes=400, path_kind=1, radius=STREAM_RADIUS)
    small = [synth.scan(oracle_lib.small_sensor(16, 360), world, synth.pose(1, STREAM_RADIUS, float(i)), 500 + i,
                        threads=cores()) for i in range(n)]
    for name, kw in _config_cases(engine):
        scans = small if name == "voxel=0" else stream[:n]
        frames = run_session(engine, scans, **kw)
        pc = dict(kw)
        want = per_call_loop(engine, scans, voxel=pc.pop("voxel", VOXEL), cfg=pc.pop("cfg", None), **pc)
        assert_matches_per_call(frames, want, name)
        assert all(f.state != slam_b200.ODOM_SKIPPED for f in frames), name
        if name == "voxel=0":
            assert all(same_bits(f.cloud, s) for f, s in zip(frames, scans))
        if name == "max_error=1e-12":
            # every delta is dropped: the pose stays the initial one while the target still advances frame by frame
            assert all(same_bits(f.pose, kw["initial_pose"]) for f in frames)
            assert any(f.icp.converged and f.icp.final_error > 1e-12 for f in frames[1:])
        if name.startswith("max_iterations"):
            k = int(name[-1])
            assert all(f.icp.num_iterations <= k for f in frames[1:]), name
    print(f"[odom-stress] {len(_config_cases(engine))} configurations match the per-call loop over {n} frames")


# ------------------------------------------------------------------ 6. output subsets
@pytest.mark.gpu
def test_every_output_subset_gives_the_all_outputs_bits(engine, stream):
    scans = stream[:6]
    ref = run_session(engine, scans)
    for mask in range(8):
        want = dict(want_cloud=bool(mask & 1), want_world_f32=bool(mask & 2), want_desc=bool(mask & 4))
        odom = slam_b200.Odometry(engine)
        for i, s in enumerate(scans):
            f, r = odom.push(s, i, **want), ref[i]
            assert (f.state, f.n_points) == (r.state, r.n_points)
            assert same_bits(f.pose, r.pose), (mask, i)
            if i > 0:
                assert same_bits(icp_bits(f.icp), icp_bits(r.icp)), (mask, i)
            for key, a, b in (("want_cloud", f.cloud, r.cloud), ("want_desc", f.desc, r.desc)):
                assert (a is None) if not want[key] else same_bits(a, b), (mask, key, i)
            if want["want_world_f32"]:
                assert np.array_equal(f.world_f32.view(np.uint32), r.world_f32.view(np.uint32)), (mask, i)
            else:
                assert f.world_f32 is None
        odom.close()


# ------------------------------------------------------------------ 7. other work on the same context between pushes
@pytest.mark.gpu
def test_interleaved_work_on_the_context_leaves_the_session_intact(engine, stream):
    n = 12
    a_scans, b_scans = stream[:n], stream[n:2 * n]
    detect = {i for i in range(4, n) if i % 2 == 0}

    def detector():
        return slam_b200.LoopClosureDetector(engine, frame_gap=3, sc_distance_threshold=1e300,
                                             icp_fitness_threshold=1e300, max_candidates=2)

    det_pc = detector()
    want = per_call_loop(engine, a_scans, det=det_pc, detect=detect)
    det_alone = detector()
    alone_a = run_session(engine, a_scans, loop=det_alone, detect=detect)
    assert_matches_per_call(alone_a, want, "alone")
    assert sum(len(f.loops) for f in alone_a) >= 1     # detect() verified and accepted candidates
    alone_b = [frame_bits(f) for f in run_session(engine, b_scans)]
    # the interleaved calls: a batch larger than any before it (the arena regrows), a large voxel grid, detect_batch on
    # the attached detector, and a second session
    big = np.concatenate(stream[24:36])
    big_off = np.r_[0, np.cumsum([len(s) for s in stream[24:36]])].astype(np.int64)
    huge = np.concatenate(stream[24:28])
    det = detector()
    a = slam_b200.Odometry(engine, loop=det)
    b = slam_b200.Odometry(engine)
    got_a, got_b = [], []
    for i in range(n):
        got_a.append(a.push(a_scans[i], i, detect=i in detect, **ALL))
        if i % 4 == 1:
            res = engine.register_batch(big, big_off, np.arange(1, 12), np.arange(0, 11), voxel=0.2)
            assert np.all(res.status == 0)
        elif i % 4 == 2:
            assert len(engine.voxel_downsample(huge, 0.2)) > 4 * SEG_CAP
        elif i % 4 == 3:
            det.detect_batch([det.size() - 1])
        got_b.append(frame_bits(b.push(b_scans[i], i, **ALL)))
    a.close()
    b.close()
    assert all(same_bits(frame_bits(x), frame_bits(y)) for x, y in zip(got_a, alone_a))
    assert all(same_bits(x, y) for x, y in zip(got_b, alone_b))
    assert det.size() == det_pc.size() == n
    assert all(same_bits(x, y) for x, y in zip(det.candidates_local(), det_pc.candidates_local()))
    for x in (det_pc, det_alone, det):
        x.close()
    print(f"[odom-stress] interleaved: {n} + {n} frames of two sessions, {sum(len(f.loops) for f in alone_a)} accepted "
          f"loop closures, identical to the sessions run alone")


# ------------------------------------------------------------------ 8. what the node publishes from the session
@pytest.mark.gpu
def test_global_map_and_occupancy_from_the_session_match_the_oracle(engine, oracle, stream):
    """slam_node.cpp:196-238 over the session's poses and downsampled clouds (skipped frames as empty clouds): the
    global map at twice the voxel size bit for bit, the occupancy cells identical."""
    scans = list(stream)
    for k in (10, 25):                      # frames below min_points: the pose repeats, the cloud is published empty
        scans.insert(k, stream[k][::200].copy())
    odom = slam_b200.Odometry(engine)
    frames = [odom.push(s, i, want_cloud=True, want_world_f32=True) for i, s in enumerate(scans)]
    odom.close()
    skipped = [i for i, f in enumerate(frames) if f.state == slam_b200.ODOM_SKIPPED]
    assert skipped == [10, 25]
    clouds = [np.zeros((0, 3)) if f.state == slam_b200.ODOM_SKIPPED else f.cloud for f in frames]
    Ts = np.stack([f.pose for f in frames])
    off = np.r_[0, np.cumsum([len(c) for c in clouds])].astype(np.int64)
    pts = np.concatenate(clouds)
    world = [oracle.transform_cloud(c, T) if len(c) else np.zeros((0, 3)) for c, T in zip(clouds, Ts)]
    for f, w in zip(frames, world):
        if f.state != slam_b200.ODOM_SKIPPED:
            assert np.array_equal(f.world_f32.view(np.uint32), w.astype(np.float32).view(np.uint32))
    ref_world = np.concatenate(world)
    gm = engine.global_map(pts, off, Ts, 2 * VOXEL)
    ref_gm, _ = oracle.voxel_downsample(ref_world, 2 * VOXEL)
    assert same_bits(gm, ref_gm)
    cells, count = engine.occupancy_cells(pts, off, Ts)
    ref_cells = oracle.occupancy_cells(pts, off, Ts)
    assert count == len(ref_cells) and np.array_equal(cells, ref_cells) and count > 1000
    print(f"[odom-stress] global map: {len(pts)} rows from {len(frames)} frames -> {len(gm)} map rows; "
          f"{count} occupancy cells")
