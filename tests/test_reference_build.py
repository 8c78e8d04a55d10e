"""The CPU oracle against the REFERENCE'S OWN SOURCES (oracle/_ref/libslam_ref.so: $REFERENCE_ROOT/slam_viz, a checkout
of the original project, compiled unmodified against oracle/eigen_standin, see oracle/build_ref.sh).

What this pins: every piece of the reference's control flow on the hot path -- the voxel hash map and its centroid
order, KD-tree build (nth_element medians) and both searches, the normal orientation rule, the ICP loop with its
doubled nearest-neighbour pass, stopping rules and history, Scan Context binning / clamping / shifting, the
loop-closure candidate filter, sort and sequential acceptance, float32 loaders.  What it does not pin is Eigen's own
floating-point kernels (eigen solver, LDLT, reductions), which the stand-in replaces with plain fp64 loops; the
tolerances below (1e-9 and tighter) are there for that substitution only.

Skipped when the library is absent: it can be built only from the original project's sources, which are not part of
this repository.
"""
import numpy as np
import pytest

import oracle_lib
import ref_lib
from conftest import rot_angle

pytestmark = pytest.mark.skipif(not ref_lib.available(), reason="oracle/_ref/libslam_ref.so not built")


@pytest.fixture(scope="module")
def ref():
    return ref_lib.Reference()


def sort_rows(x):
    return x[np.lexsort((x[:, 2], x[:, 1], x[:, 0]))]


def keys_of(rows, voxel):
    return np.floor(rows / voxel).astype(np.int64)


# ------------------------------------------------------------------ voxel grid (file_utils.cpp:148-196)
@pytest.mark.parametrize("voxel", [0.5, 0.2, 0.05])
def test_voxel_same_voxels_same_centroids(oracle, ref, synth, scene, voxel):
    raw = synth.scan(oracle_lib.small_sensor(32, 900), scene, (0.0, 0.0, 0.0), 5)
    o, okeys = oracle.voxel_downsample(raw, voxel)
    r = ref.voxel_downsample(raw, voxel)
    assert len(r) == len(o)
    # the reference emits voxels in unordered_map order and the oracle in key order: sort the rows, then the
    # centroids must agree bit for bit (same input-index summation order, same division)
    assert np.array_equal(sort_rows(r), sort_rows(o))
    assert len(np.unique(keys_of(r, voxel), axis=0)) >= len(np.unique(okeys, axis=0)) - 2  # centroid stays in its voxel


def test_voxel_nonpositive_and_empty(oracle, ref):
    pts = np.arange(12, dtype=np.float64).reshape(4, 3)
    assert np.array_equal(ref.voxel_downsample(pts, 0.0), pts)
    assert np.array_equal(ref.voxel_downsample(pts, -2.0), pts)
    assert len(ref.voxel_downsample(np.zeros((0, 3)), 0.5)) == 0
    neg = np.array([[0.6, -0.6, 0.0], [0.6000000000000001, -0.2, 1e-300], [-1e-300, 0.2, -0.0]])
    assert np.array_equal(sort_rows(ref.voxel_downsample(neg, 0.2)), sort_rows(oracle.voxel_downsample(neg, 0.2)[0]))


def test_loaders_widen_float32_records(ref, tmp_path):
    """file_utils.cpp:91-97 / 133-136: the float32 x, y, z of a record are widened to double, nothing else."""
    rng = np.random.default_rng(2)
    xyz = rng.uniform(-80, 80, (257, 3)).astype(np.float32)
    kitti = np.concatenate([xyz, rng.uniform(0, 1, (257, 1)).astype(np.float32)], axis=1)
    p = tmp_path / "000000.bin"
    kitti.tofile(p)
    assert np.array_equal(ref.load_points(str(p), True), xyz.astype(np.float64))
    ply = tmp_path / "scan.ply"
    with open(ply, "wb") as f:
        f.write(b"ply\nformat binary_little_endian 1.0\nelement vertex 257\nproperty float x\nproperty float y\n"
                b"property float z\nend_header\n")
        f.write(xyz.tobytes())
    assert np.array_equal(ref.load_points(str(ply), False), xyz.astype(np.float64))


# ------------------------------------------------------------------ KD-tree (kdtree.hpp:18-186)
@pytest.mark.parametrize("n,seed", [(1, 0), (2, 1), (7, 2), (500, 3), (4000, 4)])
def test_nearest_and_knn_match(oracle, ref, n, seed):
    rng = np.random.default_rng(seed)
    pts = rng.uniform(-10, 10, (n, 3))
    q = np.concatenate([rng.uniform(-12, 12, (300, 3)), pts[: min(n, 50)]])
    ot, rt = oracle.tree(pts), ref.tree(pts)
    oi, od = ot.nearest_batch(q)
    ri, rd = rt.nearest_batch(q)
    assert np.array_equal(oi, ri) and np.array_equal(od, rd)          # indices and squared distances bit for bit
    assert rt.nearest(q[0]) == ri[0]
    for k in (1, 5, 20):
        ok = oracle.tree(pts).k_nearest_batch(q, k)[0]
        rk = rt.k_nearest_batch(q, k)
        assert np.array_equal(ok, rk)                                  # same neighbours, same (d2, index) order


def test_knn_on_a_scan(oracle, ref, small_pair):
    pts = small_pair["a"]
    ok = oracle.tree(pts).k_nearest_batch(pts, 20)[0]
    rk = ref.tree(pts).k_nearest_batch(pts, 20)
    assert np.array_equal(ok, rk)
    assert np.array_equal(ok[:, 0], np.arange(len(pts)))               # the query itself is neighbour 0 (d2 = 0)


def test_find_correspondences(oracle, ref, small_pair):
    m, d = ref.find_correspondences(small_pair["a"], small_pair["b"])
    idx, d2 = oracle.tree(small_pair["a"]).nearest_batch(small_pair["b"])
    assert np.array_equal(m, small_pair["a"][idx]) and np.array_equal(d, np.sqrt(d2))


# ------------------------------------------------------------------ normals (icp.hpp:23-67)
@pytest.mark.parametrize("k", [20, 10, 3])
def test_normals(oracle, ref, small_pair, k):
    pts = small_pair["a"]
    on = oracle.tree(pts).estimate_normals(k)
    on = on[0] if isinstance(on, tuple) else on
    rn = ref.tree(pts).estimate_normals(k)
    # both use a Jacobi eigen solver on the same covariance; a normal is ill-defined where the two smallest
    # eigenvalues coincide, so compare up to sign where they disagree by more than rounding
    dot = np.abs(np.sum(on * rn, axis=1))
    assert np.mean(dot > 1 - 1e-9) > 0.999
    ok = np.sum(on * rn, axis=1) > 1 - 1e-9
    assert np.max(np.abs(on[ok] - rn[ok])) < 1e-7
    assert np.all(rn[:, 2] >= 0) and np.allclose(np.linalg.norm(rn, axis=1), 1.0, atol=1e-12)


def test_normals_fewer_than_three_points(oracle, ref):
    pts = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0]])
    assert np.array_equal(ref.tree(pts).estimate_normals(20), np.array([[0.0, 0.0, 1.0], [0.0, 0.0, 1.0]]))


# ------------------------------------------------------------------ solve + ICP (icp.hpp:89-258)
def test_solve_point_to_plane(oracle, ref, small_pair):
    a, b = small_pair["a"], small_pair["b"]
    tree = oracle.tree(a)
    nrm = tree.estimate_normals(20)
    nrm = nrm[0] if isinstance(nrm, tuple) else nrm
    idx, _ = tree.nearest_batch(b)
    To = oracle.solve_point_to_plane(b, a[idx], nrm[idx])
    Tr = ref.solve_point_to_plane(b, a[idx], nrm[idx])
    assert np.max(np.abs(To - Tr)) < 1e-10
    # zero motion -> the theta < 1e-10 branch (icp.hpp:130-131): exactly the identity rotation
    Tz = ref.solve_point_to_plane(a[idx], a[idx], nrm[idx])
    assert np.array_equal(Tz[:3, :3], np.eye(3)) and np.array_equal(Tz, oracle.solve_point_to_plane(a[idx], a[idx], nrm[idx]))


@pytest.mark.parametrize("cfg", [dict(), dict(max_iterations=3), dict(max_iterations=0), dict(tolerance=1e-3),
                                 dict(min_error=0.5), dict(max_iterations=30, tolerance=1e-6)])
def test_icp_loop_matches(oracle, ref, small_pair, cfg):
    o = oracle.icp_point_to_plane(small_pair["b"], small_pair["a"], **cfg)
    r = ref.icp_point_to_plane(small_pair["b"], small_pair["a"], **cfg)
    assert o["num_iterations"] == r["num_iterations"] and o["converged"] == r["converged"]
    assert len(o["error_history"]) == len(r["error_history"])
    assert np.allclose(o["error_history"], r["error_history"], rtol=0, atol=1e-9)
    assert abs(o["final_error"] - r["final_error"]) < 1e-9
    dT = o["transformation"] @ np.linalg.inv(r["transformation"])
    assert np.linalg.norm(dT[:3, 3]) < 1e-8 and rot_angle(dT[:3, :3]) < 1e-8


def planar_pair(n_side=24, dz=0.15):
    """A target whose every normal is exactly (0, 0, 1) (points on z = 0) and a source lifted off it: J^T J has rank 3
    with exact zeros on its diagonal — the case where an unpivoted LDL^T divides 0 by 0 (icp.hpp:120 uses Eigen's
    pivoted ldlt(), which leaves those components at zero)."""
    g = np.arange(n_side, dtype=np.float64) * 0.5
    xx, yy = np.meshgrid(g, g + 0.125 * (g % 1.0))
    tgt = np.stack([xx.ravel(), yy.ravel(), np.zeros(xx.size)], axis=1)
    src = tgt[::3] + np.array([0.05, -0.03, dz])
    return src, tgt


def test_icp_rank_deficient_planar_target(oracle, ref):
    src, tgt = planar_pair()
    o = oracle.icp_point_to_plane(src, tgt)
    r = ref.icp_point_to_plane(src, tgt)
    assert np.all(np.isfinite(r["transformation"])) and np.all(np.isfinite(o["transformation"]))
    assert o["num_iterations"] == r["num_iterations"] and o["converged"] == r["converged"] == 1
    assert np.allclose(o["error_history"], r["error_history"], rtol=0, atol=1e-12)
    assert np.max(np.abs(o["transformation"] - r["transformation"])) < 1e-12
    # only what the plane constrains moves: z translation (and x/y rotation), nothing in the plane
    assert abs(o["transformation"][2, 3] + 0.15) < 1e-9 and np.allclose(o["transformation"][:2, 3], 0.0, atol=1e-9)
    assert o["final_error"] < 1e-9


def test_icp_fewer_than_six_source_points(oracle, ref, small_pair):
    src = small_pair["b"][[10, 500, 900, 1500]]
    o = oracle.icp_point_to_plane(src, small_pair["a"])
    r = ref.icp_point_to_plane(src, small_pair["a"])
    # rank <= 4 with rounding-noise pivots instead of exact zeros: the step is ill-posed, so the two builds may take
    # different paths — but neither may produce a non-finite pose or error
    assert np.all(np.isfinite(r["transformation"])) and np.all(np.isfinite(o["transformation"]))
    assert np.all(np.isfinite(r["error_history"])) and np.all(np.isfinite(o["error_history"]))


def test_icp_initial_transform(oracle, ref, small_pair):
    c, s = np.cos(0.01), np.sin(0.01)
    T0 = np.array([[c, -s, 0, 0.8], [s, c, 0, 0.1], [0, 0, 1, 0.0], [0, 0, 0, 1.0]])
    o = oracle.icp_point_to_plane(small_pair["b"], small_pair["a"], T0=T0)
    r = ref.icp_point_to_plane(small_pair["b"], small_pair["a"], T0=T0)
    assert o["num_iterations"] == r["num_iterations"] and o["converged"] == r["converged"]
    assert np.max(np.abs(o["transformation"] - r["transformation"])) < 1e-8


def test_transformation_algebra(oracle, ref):
    rng = np.random.default_rng(5)
    q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    A = np.eye(4); A[:3, :3] = q * np.sign(np.linalg.det(q)); A[:3, 3] = rng.normal(size=3)
    B = np.eye(4); B[:3, 3] = [1.0, -2.0, 0.5]
    AB, Ai = ref.compose_inverse(A, B)
    assert np.allclose(AB, A @ B, atol=1e-15) and np.allclose(Ai @ A, np.eye(4), atol=1e-14)
    pts = rng.uniform(-30, 30, (100, 3))
    assert np.array_equal(ref.transform_apply(A, pts), oracle.transform_cloud(pts, A))  # P R^T + t, same op order


# ------------------------------------------------------------------ Scan Context (scan_context.hpp:24-145)
def test_scan_context_descriptor_distance_keys(oracle, ref, small_pair):
    a, b = small_pair["a"], small_pair["b"]
    da, db = oracle.sc_compute(a), oracle.sc_compute(b)
    assert np.array_equal(ref.sc_compute(a), da) and np.array_equal(ref.sc_compute(b), db)
    assert ref.sc_distance_clouds(a, b) == oracle.sc_distance(da, db)
    assert ref.sc_distance_clouds(a, a) == oracle.sc_distance(da, da)
    ring, sector = ref.sc_keys(a)
    m = da.reshape(60, 20).T                                       # column-major storage -> (ring, sector)
    assert np.allclose(ring, m.mean(axis=1), atol=1e-13) and np.allclose(sector, m.mean(axis=0), atol=1e-13)


def test_scan_context_edges(oracle, ref):
    # range limits (r > 80, r < 0.1 skipped), the atan2 seam, clamping, the -1000 floor and empty input
    pts = np.array([[80.0, 0.0, 1.0], [80.0000001, 0.0, 9.0], [0.05, 0.0, 5.0], [0.1, 0.0, 2.0], [-1.0, -0.0, 3.0],
                    [-1.0, 1e-18, 4.0], [10.0, 10.0, -1000.5], [0.0, -5.0, -999.0], [79.9999, -1e-9, 0.25]])
    assert np.array_equal(ref.sc_compute(pts), oracle.sc_compute(pts))
    assert np.array_equal(ref.sc_compute(np.zeros((0, 3))), np.zeros(1200))
    assert ref.sc_distance_clouds(np.zeros((0, 3)), pts) == 1.0     # norm < 1e-10 -> 1.0 (scan_context.hpp:137-138)


# ------------------------------------------------------------------ loop closure (loop_closure.hpp:41-149)
def test_loop_detector_sequence(oracle, ref, synth, scene):
    s = oracle_lib.small_sensor(16, 360)
    poses = [(float(i), 0.0, 0.0) for i in range(8)] + [(0.3, 0.05, 0.0), (1.2, -0.05, 0.01), (6.6, 0.0, 0.0)]
    od = oracle.loop(frame_gap=3, sc_thr=0.5, icp_thr=0.5, max_candidates=2)
    rd = ref.loop(frame_gap=3, sc_thr=0.5, icp_thr=0.5, max_candidates=2)
    found = 0
    for i, p in enumerate(poses):
        c = oracle.voxel_downsample(synth.scan(s, scene, p, 50 + i), 0.5)[0]
        od.add(c, i)
        rd.add(c, i)
        o, r = od.detect(), rd.detect()
        assert [(x["query_frame"], x["match_frame"]) for x in o] == [(x["query_frame"], x["match_frame"]) for x in r]
        for xo, xr in zip(o, r):
            assert xo["scan_context_distance"] == xr["scan_context_distance"]
            assert abs(xo["icp_fitness"] - xr["icp_fitness"]) < 1e-9
            assert np.max(np.abs(xo["transform"] - xr["transform"])) < 1e-8
        found += len(r)
    assert found > 0 and rd.size() == len(poses)
    rd.clear()
    assert rd.size() == 0 and rd.detect() == []


# ------------------------------------------------------------------ exact ties and many random shapes
def test_exact_ties_on_a_lattice(oracle, ref):
    """On exact distance ties the reference returns whichever minimiser its traversal meets first (kdtree.hpp:125,160
    with nth_element's unspecified partition); the oracle and the engine return the smallest index.  Both must agree
    on the DISTANCES bit for bit, the reference's pick must be a true minimiser, and the oracle's the first of them."""
    rng = np.random.default_rng(9)
    g = np.arange(-4, 5, dtype=np.float64)
    pts = np.stack(np.meshgrid(g, g, g, indexing="ij"), axis=-1).reshape(-1, 3)
    pts = pts[rng.permutation(len(pts))]
    q = np.concatenate([rng.integers(-5, 6, (200, 3)).astype(np.float64) + 0.5, pts[:50]])  # cell centres: 8-way ties
    ot, rt = oracle.tree(pts), ref.tree(pts)
    oi, od = ot.nearest_batch(q)
    ri, rd = rt.nearest_batch(q)
    assert np.array_equal(od, rd)
    d_all = ((pts[None, :, :] - q[:, None, :]) ** 2).sum(axis=2)
    assert np.array_equal(d_all[np.arange(len(q)), ri], rd)                    # the reference's pick is a minimiser
    assert np.array_equal(oi, np.argmax(d_all == d_all.min(axis=1, keepdims=True), axis=1))  # oracle: first minimiser
    for k in (4, 20):
        ok, okd = ot.k_nearest_batch(q, k)
        rk = rt.k_nearest_batch(q, k)
        rkd = d_all[np.arange(len(q))[:, None], rk]
        assert np.array_equal(okd, rkd)                                         # same multiset of distances, ascending
        inside = okd[:, -1:] > okd                                              # strictly inside the k-th distance:
        for row in range(len(q)):                                               # those neighbours are forced
            assert set(ok[row][inside[row]]) <= set(rk[row])


@pytest.mark.parametrize("seed", range(6))
def test_random_shapes_nearest_and_knn(oracle, ref, seed):
    rng = np.random.default_rng(100 + seed)
    for _ in range(12):
        n = int(rng.integers(1, 400))
        kind = rng.integers(0, 3)
        if kind == 0:
            pts = rng.normal(size=(n, 3)) * rng.uniform(0.1, 50)
        elif kind == 1:   # thin slab: one axis nearly degenerate (the split axis cycles regardless, kdtree.hpp:90)
            pts = rng.uniform(-30, 30, (n, 3)) * np.array([1.0, 1.0, 1e-6])
        else:             # clustered
            pts = rng.normal(size=(n, 3)) * 0.05 + rng.integers(-3, 4, (n, 1)) * 10.0
        q = np.concatenate([pts[rng.integers(0, n, 20)] + rng.normal(size=(20, 3)) * 0.3, rng.uniform(-60, 60, (20, 3))])
        ot, rt = oracle.tree(pts), ref.tree(pts)
        oi, od = ot.nearest_batch(q)
        ri, rd = rt.nearest_batch(q)
        assert np.array_equal(oi, ri) and np.array_equal(od, rd)
        k = int(rng.choice([1, 3, 10, 20, 32]))
        assert np.array_equal(ot.k_nearest_batch(q, k)[0], rt.k_nearest_batch(q, k))


@pytest.mark.parametrize("voxel,scale", [(0.01, 5.0), (2.0, 500.0), (0.3, 80.0)])
def test_voxel_grid_scales_and_signs(oracle, ref, voxel, scale):
    rng = np.random.default_rng(int(voxel * 1000))
    pts = (rng.uniform(-scale, scale, (5000, 3))).astype(np.float32).astype(np.float64)
    pts[:50] = pts[50:100] + np.float32(1e-4)     # near-duplicates share voxels
    o, _ = oracle.voxel_downsample(pts, voxel)
    r = ref.voxel_downsample(pts, voxel)
    assert np.array_equal(sort_rows(o), sort_rows(r))


# ------------------------------------------------------------------ property-based (hypothesis), small sizes
from hypothesis import given, settings, strategies as st  # noqa: E402
from hypothesis.extra import numpy as hnp  # noqa: E402

_coords = st.floats(min_value=-200.0, max_value=200.0, allow_nan=False, allow_infinity=False, width=32)


@settings(max_examples=60, deadline=None, derandomize=True)
@given(pts=hnp.arrays(np.float32, st.tuples(st.integers(1, 120), st.just(3)), elements=_coords),
       voxel=st.sampled_from([0.05, 0.2, 0.5, 1.0, 7.5]))
def test_property_voxel_grid(pts, voxel):
    """Any float32 cloud (duplicates, zeros, negative zero, denormals included): same voxel set, same centroids."""
    o = _ORACLE.voxel_downsample(pts.astype(np.float64), voxel)[0]
    r = _REF.voxel_downsample(pts.astype(np.float64), voxel)
    assert np.array_equal(sort_rows(o), sort_rows(r))


@settings(max_examples=60, deadline=None, derandomize=True)
@given(pts=hnp.arrays(np.float64, st.tuples(st.integers(1, 80), st.just(3)),
                      elements=st.floats(-50, 50, allow_nan=False, allow_infinity=False)),
       q=hnp.arrays(np.float64, st.tuples(st.integers(1, 20), st.just(3)),
                    elements=st.floats(-60, 60, allow_nan=False, allow_infinity=False)),
       k=st.integers(1, 32))
def test_property_search_distances(pts, q, k):
    """Arbitrary clouds (exact duplicates and ties allowed): nearest and k-nearest DISTANCES agree bit for bit; indices
    agree wherever the distance is not shared with another point."""
    ot, rt = _ORACLE.tree(pts), _REF.tree(pts)
    oi, od = ot.nearest_batch(q)
    ri, rd = rt.nearest_batch(q)
    assert np.array_equal(od, rd)
    d_all = ((pts[None, :, 0] - q[:, None, 0]) ** 2 + (pts[None, :, 1] - q[:, None, 1]) ** 2) + (pts[None, :, 2] - q[:, None, 2]) ** 2
    unique_min = (d_all == d_all.min(axis=1, keepdims=True)).sum(axis=1) == 1
    assert np.array_equal(oi[unique_min], ri[unique_min])
    ok, okd = ot.k_nearest_batch(q, k)
    rk = rt.k_nearest_batch(q, k)
    m = min(k, len(pts))
    rkd = np.take_along_axis(d_all, np.clip(rk[:, :m], 0, None), axis=1)
    assert np.array_equal(okd[:, :m], rkd) and np.all(rk[:, m:] == -1) and np.all(ok[:, m:] == -1)


_ORACLE = oracle_lib.Oracle()
_REF = ref_lib.Reference() if ref_lib.available() else None
