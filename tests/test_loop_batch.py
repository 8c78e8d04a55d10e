"""Loop-closure detection over a whole sequence in one call (sb_loop_add_frames, sb_loop_candidates_batch,
sb_loop_detect_batch): the result for query entry q is what detect() returns right after entry q was added
(loop_closure.hpp:53-126, driven as slam_node.cpp:159-167 drives it)."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import oracle_lib
from conftest import rot_angle

ROOT = oracle_lib.ROOT
N_SEQ = 120


def seq_pose(i):
    """1 m steps out along x for 60 frames, then back 0.2 m to the side: frame 60 + k revisits frame 59 - k."""
    return (float(i), 0.0, 0.0) if i < 60 else (float(119 - i), 0.2, 0.0)


@pytest.fixture(scope="module")
def sequence(oracle, synth, scene):
    s = oracle_lib.small_sensor(16, 360)
    clouds = [oracle.voxel_downsample(synth.scan(s, scene, seq_pose(i), 300 + i), 0.5)[0] for i in range(N_SEQ)]
    off = np.zeros(N_SEQ + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(c) for c in clouds])
    return clouds, np.vstack(clouds), off


def same_loops(got, want):
    assert [(r["query_frame"], r["match_frame"]) for r in got] == [(r["query_frame"], r["match_frame"]) for r in want]
    for a, b in zip(got, want):
        assert a["scan_context_distance"] == b["scan_context_distance"]
        assert a["icp_fitness"] == b["icp_fitness"]
        assert np.array_equal(a["transform"], b["transform"])


@pytest.mark.gpu
@pytest.mark.parametrize("max_candidates", [2, 4])
def test_sequence_matches_per_frame_detect(engine, oracle, sequence, max_candidates):
    import slam_b200
    clouds, xyz, off = sequence
    kw = dict(frame_gap=10, sc_distance_threshold=0.5, icp_fitness_threshold=0.3, max_candidates=max_candidates)
    one = slam_b200.LoopClosureDetector(engine, **kw)
    odet = oracle.loop(frame_gap=10, sc_thr=0.5, icp_thr=0.3, max_candidates=max_candidates)
    queries = [i for i in range(N_SEQ) if i % 5 == 0 and i > 10]
    oracle_queries = {20, 75, 100}
    cand_one, det_one, det_orc = {}, {}, {}
    for i, c in enumerate(clouds):
        one.addFrame(c, i)
        odet.add(c, i)
        if i in queries:
            cand_one[i] = one.candidates_local()
            det_one[i] = one.detect()
            if i in oracle_queries:
                det_orc[i] = odet.detect()
    bulk = slam_b200.LoopClosureDetector(engine, **kw)
    bulk.addFrames(xyz, off, np.arange(N_SEQ))
    lists, counts = bulk.candidates_batch(queries)
    got = bulk.detect_batch(queries)
    for j, q in enumerate(queries):
        d1, e1 = cand_one[q]
        assert counts[j] == len(e1)
        assert np.array_equal(lists[j][0], d1[:32]) and np.array_equal(lists[j][1], e1[:32])
        same_loops(got[j], det_one[q])
        assert all(r["query_frame"] == q for r in got[j])
    for q, want in det_orc.items():   # tolerances of test_loop_detector_matches_oracle
        g = got[queries.index(q)]
        assert [(r["query_frame"], r["match_frame"]) for r in g] == [(r["query_frame"], r["match_frame"]) for r in want]
        for rg, ro in zip(g, want):
            assert rg["scan_context_distance"] == ro["scan_context_distance"]
            assert abs(rg["icp_fitness"] - ro["icp_fitness"]) < 1e-6
            dT = rg["transform"] @ np.linalg.inv(ro["transform"])
            assert np.linalg.norm(dT[:3, 3]) < 1e-4 and rot_angle(dT[:3, :3]) < 1e-5
    assert any(len(g) > 0 for g in got) and any(len(g) == 0 for g in got)
    # the batch call leaves the detector as it was
    same_loops(bulk.detect(), one.detect())
    assert all(np.array_equal(a, b) for a, b in zip(bulk.candidates_local(), one.candidates_local()))


@pytest.mark.gpu
def test_walk_past_the_short_list(engine, oracle, synth, scene):
    """More than 32 candidates and the best 32 all fail ICP (decoys: clouds of another place with the descriptors
    closest to the query's), verify_chunk 3 (does not divide 32): the walk must go on at rank 32 of the full list."""
    import sharding
    import slam_b200
    s = oracle_lib.small_sensor(16, 360)
    cloud = lambda p, seed: oracle.voxel_downsample(synth.scan(s, scene, p, seed), 0.5)[0]
    qc = cloud((0.0, 0.0, 0.0), 900)
    base = engine.sc_compute(qc)
    rng = np.random.default_rng(5)
    det = slam_b200.LoopClosureDetector(engine, frame_gap=10, sc_distance_threshold=1e300, icp_fitness_threshold=0.3,
                                        max_candidates=2, verify_chunk=3)
    n_decoy, n_true = 40, 3
    for i in range(n_decoy):   # another place, 40 m away, with a near copy of the query's descriptor
        det.addFrame(cloud((40.0 + 0.5 * (i % 4), 0.0, 0.0), 910 + i), i,
                     desc=base + rng.uniform(0, 0.01, 1200) * (base != 0))
    for i in range(n_true):    # the same place, with a descriptor further away
        det.addFrame(cloud((0.3 * (i + 1), 0.1, 0.0), 960 + i), n_decoy + i,
                     desc=base + rng.uniform(0, 2.0, 1200) * (base != 0))
    det.addFrame(qc, 100)
    q = n_decoy + n_true
    d, e = det.candidates_local(capacity=4096)
    assert len(e) == n_decoy + n_true and set(e[32:]) >= set(range(n_decoy, q))
    res, conv = det.verify_entries(e, d)
    acc = sharding.accept_in_order(e, conv, [r["icp_fitness"] for r in res], 0.3, 2)
    assert acc and min(list(e).index(a) for a in acc) >= 32
    got = det.detect_batch([q])[0]
    assert [r["match_frame"] for r in got] == acc   # frame = entry here
    for r in got:
        ref = res[list(e).index(r["match_frame"])]
        assert r["query_frame"] == 100 and r["icp_fitness"] == ref["icp_fitness"]
        assert np.array_equal(r["transform"], ref["transform"])


@pytest.mark.gpu
@pytest.mark.parametrize("with_desc", [False, True])
def test_bulk_add_equals_per_frame_add(engine, sequence, with_desc):
    import slam_b200
    clouds, xyz, off = sequence
    n = 30
    frames = np.arange(n) * 2 + 7
    descs = np.stack([engine.sc_compute(c) for c in clouds[:n]]) if with_desc else None
    kw = dict(frame_gap=8, sc_distance_threshold=0.6, icp_fitness_threshold=0.5)

    def one_by_one(**extra):
        d = slam_b200.LoopClosureDetector(engine, **kw, **extra)
        for i in range(n):
            d.addFrame(clouds[i], int(frames[i]), desc=None if descs is None else descs[i])
        return d

    def bulk(**extra):
        d = slam_b200.LoopClosureDetector(engine, **kw, **extra)
        for a, b in ((0, 11), (11, n)):   # two calls: the second starts after a guest entry on world 2
            d.addFrames(xyz[off[a]:off[b]], off[a:b + 1] - off[a], frames[a:b],
                        None if descs is None else descs[a:b])
        return d

    a, b = one_by_one(), bulk()
    assert a.size() == b.size() == n
    for x, y in zip(a.candidates_local(), b.candidates_local()):
        assert np.array_equal(x, y)
    same_loops(b.detect(), a.detect())
    # world = 2 emulated on one GPU, as test_loop_sharded_candidates_merge: same local lists and verification per rank
    for r in (0, 1):
        a, b = one_by_one(rank=r, world=2), bulk(rank=r, world=2)
        assert a.size() == b.size() == n
        da, ea = a.candidates_local()
        db, eb = b.candidates_local()
        assert np.array_equal(da, db) and np.array_equal(ea, eb)
        if len(ea):
            ra, ca = a.verify_entries(ea[:3], da[:3])
            rb, cb = b.verify_entries(eb[:3], db[:3])
            assert np.array_equal(ca, cb)
            for x, y in zip(ra, rb):
                assert x["query_frame"] == y["query_frame"] == frames[-1]
                assert np.array_equal(x["transform"], y["transform"])


@pytest.mark.gpu
def test_query_groups_bit_equal_to_single_query_search(engine):
    """Q x D large enough that the distance matrix runs in several groups (32 MB each): sampled rows equal the
    one-query search on the truncated database, and the selection equals a lexsort after the gap and threshold."""
    import slam_b200
    rng = np.random.default_rng(11)
    n = 4000
    base = np.where(rng.uniform(size=(40, 60, 20)) < 0.35, rng.uniform(-1.7, 9.0, (40, 60, 20)), 0.0)
    db = base[rng.integers(0, 40, n)] + np.where(rng.uniform(size=(n, 60, 20)) < 0.05, rng.normal(0, 0.5, (n, 60, 20)), 0.0)
    db = np.stack([np.roll(d, int(sft), axis=0) for d, sft in zip(db, rng.integers(0, 60, n))]).reshape(n, -1)
    gap = 5
    thr = float(np.median(engine.sc_distance_batch(db[n - 1], db[:n - 1])))
    det = slam_b200.LoopClosureDetector(engine, frame_gap=gap, sc_distance_threshold=thr)
    pts = rng.uniform(-20, 20, (n * 8, 3))
    det.addFrames(pts, np.arange(n + 1) * 8, np.arange(n), db)
    queries = np.arange(1, n)
    rows = (32 << 20) // (8 * int(queries[-1])) // 8 * 8
    assert len(queries) > 2 * rows   # at least three groups
    lists, counts = det.candidates_batch(queries, k=32)
    sample = sorted({0, 1, gap, rows - 1, rows, rows + 1, 2 * rows - 1, 2 * rows, len(queries) - 1} |
                    set(rng.integers(0, len(queries), 6).tolist()))
    for j in sample:
        q = int(queries[j])
        d = engine.sc_distance_batch(db[q], db[:q])
        e = np.arange(q)
        keep = (q - e >= gap) & (d < thr)
        order = np.lexsort((e[keep], d[keep]))
        assert counts[j] == keep.sum()
        assert np.array_equal(lists[j][1], e[keep][order][:32])
        assert np.array_equal(lists[j][0], d[keep][order][:32])


@pytest.mark.gpu
def test_edges(engine, sequence):
    import slam_b200
    clouds, xyz, off = sequence
    n = 40
    det = slam_b200.LoopClosureDetector(engine, frame_gap=10, sc_distance_threshold=0.6, icp_fitness_threshold=0.5)
    det.addFrames(xyz[:off[n]], off[:n + 1], np.arange(n))
    before = det.detect(), det.candidates_local()
    assert det.detect_batch([0]) == [[]]
    lists, counts = det.candidates_batch([0, 5])
    assert list(counts) == [0, 0] and all(len(x[1]) == 0 for x in lists)
    far = slam_b200.LoopClosureDetector(engine, frame_gap=1000, sc_distance_threshold=0.6)
    far.addFrames(xyz[:off[n]], off[:n + 1], np.arange(n))
    assert far.detect_batch([10, 20, 39]) == [[], [], []]
    assert list(far.candidates_batch([10, 39])[1]) == [0, 0]
    none = slam_b200.LoopClosureDetector(engine, frame_gap=10, sc_distance_threshold=0.6, max_candidates=0)
    none.addFrames(xyz[:off[n]], off[:n + 1], np.arange(n))
    assert none.detect_batch([20, 39]) == [[], []]
    for bad in ([5, 5], [7, 3], [-1], [n], [0, n + 3]):
        with pytest.raises(slam_b200.SlamB200Error) as ex:
            det.detect_batch(bad)
        assert ex.value.status == 1
        with pytest.raises(slam_b200.SlamB200Error) as ex:
            det.candidates_batch(bad)
        assert ex.value.status == 1
    for k in (0, 33):
        with pytest.raises(slam_b200.SlamB200Error) as ex:
            det.candidates_batch([5], k=k)
        assert ex.value.status == 1
    w2 = slam_b200.LoopClosureDetector(engine, frame_gap=10, rank=0, world=2)
    w2.addFrames(xyz[:off[n]], off[:n + 1], np.arange(n))
    for call in (lambda: w2.detect_batch([20]), lambda: w2.candidates_batch([20])):
        with pytest.raises(slam_b200.SlamB200Error) as ex:
            call()
        assert ex.value.status == 1
    det.detect_batch(list(range(12, n, 3)))
    same_loops(det.detect(), before[0])
    assert all(np.array_equal(a, b) for a, b in zip(det.candidates_local(), before[1]))


def build_mirror_test(out_dir):
    """tests/cpp/loop_batch_test.cpp over the mirror headers, linked like tests/cpp/build.sh links host_api_test."""
    oracle_lib.Synth()  # builds libsynth.so if needed
    lib = os.path.join(ROOT, "lidar-slam-from-scratch_b200")
    exe = os.path.join(out_dir, "loop_batch_test")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-Wno-unused-function", "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(lib, "host"), os.path.join(ROOT, "tests", "cpp", "loop_batch_test.cpp"),
                           "-o", exe, "-L" + lib, "-lslam_b200", "-L" + os.path.join(ROOT, "synth"), "-lsynth",
                           "-Wl,-rpath," + lib, "-Wl,-rpath," + os.path.join(ROOT, "synth")])
    return exe


def test_mirror_sequence_extensions_compile():
    with tempfile.TemporaryDirectory() as d:
        assert os.path.exists(build_mirror_test(d))


@pytest.mark.gpu
def test_mirror_sequence_extensions_match_per_frame_detect():
    with tempfile.TemporaryDirectory() as d:
        p = subprocess.run([build_mirror_test(d)], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "all checks passed" in p.stdout
