"""The drop-in boundary, tested the way INTEGRATION.md section 1 describes it.

CPU: the reference's UNMODIFIED slam_viz/src/ros/slam_node.cpp and src/core/file_utils.cpp compile with the mirror
directory (lidar-slam-from-scratch_b200/host) in front of the reference's include directory and link against
libslam_b200.so; the node's voxel_downsample binds to the GPU entry point; the node's call sites also compile in the
mirror's no-Eigen branch (tests/cpp/call_sites_test.cpp).  ROS 2 is tests/cpp/ros_stubs, Eigen is the oracle's
stand-in, slam::PoseGraph is a GTSAM-free test double (tests/cpp/pose_graph_double.cpp).

GPU: that binary runs the node's own process_frame loop (slam_node.cpp:95-175) over synthetic PLY frames on the
engine, and what it hands to its pose graph (SURVEY.md 8f N4) equals the batch path's sb_odometry_factors.

Both need the original project's sources, which are not part of this repository: REFERENCE_ROOT names a checkout of it,
and without one these tests skip."""
import json
import os
import subprocess

import numpy as np
import pytest

import oracle_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPP = os.path.join(ROOT, "tests", "cpp")
EXE = os.path.join(CPP, "slam_node_dropin")
# the original project's checkout (its slam_viz/ directory below it): REFERENCE_ROOT, unset where it is absent
REF = os.path.join(os.environ["REFERENCE_ROOT"], "slam_viz") if os.environ.get("REFERENCE_ROOT") else None


HAVE_REF = REF is not None and os.path.exists(os.path.join(REF, "src", "ros", "slam_node.cpp"))
NEEDS_REF = "needs the original project's sources: REFERENCE_ROOT names its checkout"


def build():
    oracle_lib.Oracle(), oracle_lib.Synth()
    import slam_b200
    slam_b200.load_library()
    subprocess.check_call(["sh", os.path.join(CPP, "build.sh")])


def node_binary():
    """tests/cpp/slam_node_dropin, built here from the original project's sources; skips the test without them."""
    if not HAVE_REF:
        pytest.skip(NEEDS_REF)
    build()
    return EXE


@pytest.mark.skipif(not HAVE_REF, reason=NEEDS_REF)
def test_reference_node_compiles_and_links_against_the_mirror():
    build()  # raises if slam_node.cpp / file_utils.cpp / call_sites_test.cpp do not compile or the link fails
    assert os.path.exists(EXE)
    sym = subprocess.run(["nm", "-C", EXE], capture_output=True, text=True, check=True).stdout
    # the node calls the GPU voxel grid (inline namespace b200_impl -> sb_voxel_downsample) ...
    assert "slam::b200_impl::voxel_downsample(" in sym
    assert " U sb_voxel_downsample" in sym and " U sb_icp_point_to_plane" in sym and " U sb_loop_detect" in sym
    # ... the loaders are the reference's own (file_utils.cpp), whose CPU voxel grid is a separate, unused symbol
    for name in ("slam::load_ply(", "slam::load_bin(", "slam::discover_frames(", "slam::extract_timestamp("):
        assert any(l.split()[1:2] == ["T"] and name in l for l in sym.splitlines()), name
    assert any(" T slam::voxel_downsample(" in l for l in sym.splitlines())
    for obj in ("call_sites_noeigen.o", "call_sites_eigenapi.o"):
        assert os.path.exists(os.path.join(CPP, "obj", obj))


def test_node_binary_refuses_to_run_without_a_gpu(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu test")
    node_binary()
    write_ply(tmp_path / "000000.ply", np.zeros((8, 3), np.float32))
    env = dict(os.environ, SLAM_PARAM_data_dir=str(tmp_path), SLAM_STUB_VERBOSE="1")
    p = subprocess.run([EXE], capture_output=True, text=True, env=env)
    assert "no usable sm_100a device" in p.stderr  # slam_node.cpp:343-347 catches and logs it


def write_ply(path, xyz32):
    """binary PLY with float32 x, y, z + intensity, the layout tools/convert_to_ply.cpp:36-67 writes"""
    rec = np.zeros((len(xyz32), 4), dtype="<f4")
    rec[:, :3] = xyz32
    with open(path, "wb") as f:
        f.write(("ply\nformat binary_little_endian 1.0\nelement vertex %d\nproperty float x\nproperty float y\n"
                 "property float z\nproperty float intensity\nend_header\n" % len(xyz32)).encode())
        f.write(rec.tobytes())


@pytest.mark.gpu
def test_reference_node_runs_on_the_engine_and_hands_off_the_same_factors(tmp_path, synth, engine):
    node_binary()
    scene = synth.scene(5, n_boxes=400)
    s = oracle_lib.small_sensor(32, 600)
    n_frames = 7
    scans = [synth.scan(s, scene, (1.0 * i, 0.05 * i, 0.004 * i), 40 + i) for i in range(n_frames)]
    for i, sc in enumerate(scans):
        assert np.array_equal(sc.astype(np.float32).astype(np.float64), sc)  # float32-born, like a PLY file's records
        write_ply(tmp_path / ("%06d.ply" % (1000 + i)), sc.astype(np.float32))
    out = tmp_path / "factors.json"
    env = dict(os.environ, SLAM_PARAM_data_dir=str(tmp_path), SLAM_STUB_TICKS=str(n_frames + 2),
               SLAM_DOUBLE_OUT=str(out), SLAM_STUB_VERBOSE="1")
    p = subprocess.run([EXE], capture_output=True, text=True, env=env, timeout=600)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "Error:" not in p.stderr, p.stderr
    assert "Processing complete!" in p.stderr
    rec = json.loads(out.read_text())
    assert rec["num_poses"] == n_frames and rec["num_loop_closures"] == 0
    prior, odo = rec["factors"][0], rec["factors"][1:]
    assert prior["kind"] == 0 and prior["sigmas"] == [0.001] * 6  # pose_graph.hpp:31-32
    assert [f["kind"] for f in odo] == [1] * (n_frames - 1)

    # the same frames as ONE batch through the C ABI, then sb_odometry_factors / sb_odometry_poses
    off = np.cumsum([0] + [len(x) for x in scans]).astype(np.int64)
    src, tgt = np.arange(1, n_frames, dtype=np.int32), np.arange(0, n_frames - 1, dtype=np.int32)
    res = engine.register_batch(np.vstack(scans), off, src, tgt, voxel=0.5)
    fac = engine.odometry_factors(res, first_frame=0, max_error=1.0)
    poses = engine.odometry_poses(res, max_error=1.0)
    for i, f in enumerate(odo):
        assert (f["from"], f["to"]) == (i, i + 1) == (int(fac["from"][i]), int(fac["to"][i]))
        np.testing.assert_allclose(np.array(f["relative"]).reshape(4, 4), fac["relative"][i], rtol=0, atol=1e-12)
        scale = 1.0 + 10.0 * float(res[i].final_error)  # pose_graph.cpp:88
        assert abs(fac["noise_scale"][i] - scale) < 1e-15
        np.testing.assert_allclose(f["sigmas"], [0.01 * scale] * 3 + [0.05 * scale] * 3, rtol=1e-12)
    # the back end's initial estimates (pose_graph.cpp:107-113) are the odometry chain of slam_node.cpp:142
    for i, pm in enumerate(rec["poses"]):
        np.testing.assert_allclose(np.array(pm).reshape(4, 4), poses[i], rtol=0, atol=1e-10)
    # and the motion is the one the scans were generated with (1 m per frame along x)
    step = np.linalg.norm(poses[-1][:3, 3]) / (n_frames - 1)
    assert 0.9 < step < 1.1
