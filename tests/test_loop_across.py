"""Loop closures across detectors (sb_loop_candidates_across, sb_loop_detect_across, slam_b200.candidates_across /
detect_across): query (d, e) gets detect()'s rule (loop_closure.hpp:75-122) over the entries of every other detector,
without a frame gap.  Every result must equal, bit for bit, sb_loop_candidates_batch / sb_loop_detect_batch on a
scratch detector that holds the other detectors' entries in detector order, with their own frame indices, and then the
query clouds at frame 2^30 with frame_gap 1 (queries appended together exclude each other through the gap)."""
import ctypes as C
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "lidar-slam-from-scratch_b200", "python"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import oracle_lib  # noqa: E402
import slam_b200  # noqa: E402

Q_FRAME = 1 << 30
KW = dict(sc_distance_threshold=0.5, icp_fitness_threshold=0.3, max_candidates=3)


# ------------------------------------------------------------------ CPU
def test_symbols_load():
    lib = slam_b200.load_library()
    assert hasattr(lib, "sb_loop_candidates_across") and hasattr(lib, "sb_loop_detect_across")
    assert "sb_loop_candidates_across" in slam_b200.SYMBOLS and "sb_loop_detect_across" in slam_b200.SYMBOLS


def test_null_and_negative_arguments_are_refused_and_no_queries_is_a_no_op():
    lib = slam_b200.load_library()
    i32 = C.POINTER(C.c_int32)
    one = (C.c_int32 * 1)(0)
    dist = (C.c_double * 32)()
    out = (C.c_int32 * 32)()
    cand = lib.sb_loop_candidates_across
    det = lib.sb_loop_detect_across
    # n_queries == 0: nothing to do, nothing read
    assert cand(None, 0, None, None, 0, 32, None, None, None, None) == 0
    assert det(None, 0, None, None, 0, None, None, None) == 0
    # negative counts, k out of range, null arrays
    assert cand(None, -1, None, None, 0, 32, None, None, None, None) == 1
    assert cand(None, 1, None, None, -1, 32, None, None, None, None) == 1
    assert det(None, -1, None, None, 0, None, None, None) == 1
    assert det(None, 1, None, None, -1, None, None, None) == 1
    for k in (0, 33):
        assert cand(None, 0, None, None, 0, k, None, None, None, None) == 1
    assert cand(None, 1, C.cast(one, i32), C.cast(one, i32), 1, 32, dist, out, out, out) == 1
    assert det(None, 1, C.cast(one, i32), C.cast(one, i32), 1, None, out, out) == 1
    nulls = (slam_b200._P * 1)(None)
    assert cand(nulls, 1, C.cast(one, i32), C.cast(one, i32), 1, 32, dist, out, out, out) == 1
    assert det(nulls, 1, C.cast(one, i32), C.cast(one, i32), 1, None, out, out) == 1
    assert cand(nulls, 0, C.cast(one, i32), C.cast(one, i32), 1, 32, dist, out, out, out) == 1


def test_mirror_detect_across_compiles():
    """slam::b200::detectAcross over the mirror headers (compile only)."""
    prog = r'''
#include "slam_viz/core/loop_closure.hpp"
std::vector<std::vector<slam::b200::AcrossLoop>> f(std::vector<slam::LoopClosureDetector*>& d,
                                                   const std::vector<std::pair<int, int>>& q) {
  return slam::b200::detectAcross(d, q);
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
class Stream:
    """What one detector holds: its clouds (host rows), descriptors and frame indices, in entry order."""

    def __init__(self, clouds, frames, descs=None):
        self.clouds, self.frames, self.descs = list(clouds), list(frames), descs

    def csr(self):
        off = np.zeros(len(self.clouds) + 1, dtype=np.int64)
        off[1:] = np.cumsum([len(c) for c in self.clouds])
        xyz = np.vstack(self.clouds) if self.clouds else np.zeros((0, 3))
        return xyz, off

    def detector(self, engine, **kw):
        det = slam_b200.LoopClosureDetector(engine, **kw)
        if self.clouds:
            xyz, off = self.csr()
            det.addFrames(xyz, off, self.frames, self.descs)
        return det


def scratch(engine, streams, qd, queries, kw):
    """The scratch detector of query detector qd: the other streams in order, then the query entries at frame 2^30.
    Returns it, the entry of its first query and the (db, entry) of each of its database entries."""
    det = slam_b200.LoopClosureDetector(engine, frame_gap=1, **kw)
    owner = []
    for d, s in enumerate(streams):
        if d == qd or not s.clouds:
            continue
        xyz, off = s.csr()
        det.addFrames(xyz, off, s.frames, s.descs)
        owner += [(d, e) for e in range(len(s.clouds))]
    qs = Stream([streams[qd].clouds[e] for e in queries], [Q_FRAME] * len(queries),
                None if streams[qd].descs is None else streams[qd].descs[list(queries)])
    xyz, off = qs.csr()
    det.addFrames(xyz, off, qs.frames, qs.descs)
    return det, len(owner), owner


def reference(engine, streams, queries, kw, k=32):
    """Per query: scratch candidates (dist, db, entry), count, and detect results with match_db, from the scratch
    detectors of the query detectors."""
    out = [None] * len(queries)
    for qd in sorted({d for d, _ in queries}):
        idx = [i for i, (d, _) in enumerate(queries) if d == qd]
        det, first, owner = scratch(engine, streams, qd, [queries[i][1] for i in idx], kw)
        q = list(range(first, first + len(idx)))
        lists, counts = det.candidates_batch(q, k=k)
        loops = det.detect_batch(q)
        for j, i in enumerate(idx):
            d, e = lists[j]
            dbs = np.array([owner[x][0] for x in e], dtype=np.int32)
            ents = np.array([owner[x][1] for x in e], dtype=np.int32)
            for r in loops[j]:
                assert r["query_frame"] == Q_FRAME
            out[i] = (d, dbs, ents, int(counts[j]), loops[j])
    return out


def same_as_reference(engine, dbs, streams, queries, kw, frame_db):
    lists, counts = slam_b200.candidates_across(dbs, queries)
    got = slam_b200.detect_across(dbs, queries)
    ref = reference(engine, streams, queries, kw)
    for i, (qd, qe) in enumerate(queries):
        d, db, ent, cnt, loops = ref[i]
        assert counts[i] == cnt
        assert np.array_equal(lists[i][0], d) and np.array_equal(lists[i][1], db) and np.array_equal(lists[i][2], ent)
        assert len(got[i]) == len(loops)
        for a, b in zip(got[i], loops):
            assert a["query_frame"] == streams[qd].frames[qe]
            assert a["match_frame"] == b["match_frame"] and a["match_db"] == frame_db(b["match_frame"])
            assert a["scan_context_distance"] == b["scan_context_distance"]
            assert a["icp_fitness"] == b["icp_fitness"]
            assert np.array_equal(a["transform"], b["transform"])
    return lists, counts, got


# ------------------------------------------------------------------ GPU
SEG = [  # (first x, lateral y, frames): detector d drives 1 m steps from x0 at lateral offset y, same heading
    (0.0, 0.0, 24), (12.0, 0.25, 24), (30.0, -0.2, 20), (20.0, 0.1, 8)]


@pytest.fixture(scope="module")
def streams(oracle, synth, scene):
    s = oracle_lib.small_sensor(16, 360)
    out = []
    for d, (x0, y, n) in enumerate(SEG):
        clouds = [oracle.voxel_downsample(synth.scan(s, scene, (x0 + i, y, 0.0), 500 + 100 * d + i), 0.5)[0]
                  for i in range(n)]
        out.append(Stream(clouds, [1000 * d + i for i in range(n)]))
    return out


@pytest.mark.gpu
def test_equivalence_with_scratch_detectors(engine, streams):
    dbs = [s.detector(engine, frame_gap=50, **KW) for s in streams]
    queries = [(1, 5), (0, 20), (2, 3), (0, 2), (3, 4), (1, 20), (2, 15), (0, 20), (1, 0), (3, 0), (0, 14)]
    _, counts, got = same_as_reference(engine, dbs, streams, queries, KW, lambda f: f // 1000)
    assert any(len(g) > 0 for g in got) and any(len(g) == 0 for g in got)
    assert any(r["match_db"] != qd for g, (qd, _) in zip(got, queries) for r in g)
    assert all(r["match_db"] != qd for g, (qd, _) in zip(got, queries) for r in g)
    assert [r["match_frame"] for r in got[1]] == [r["match_frame"] for r in got[7]]   # the repeated query
    assert all(np.array_equal(a["transform"], b["transform"]) for a, b in zip(got[1], got[7]))


@pytest.mark.gpu
def test_matches_oracle(engine, oracle, streams):
    """Three queries against oracle.loop on the scratch concatenation (test_loop_batch.py's tolerances)."""
    from conftest import rot_angle
    dbs = [s.detector(engine, frame_gap=50, **KW) for s in streams]
    queries = [(1, 5), (0, 20), (2, 3)]
    got = slam_b200.detect_across(dbs, queries)
    for (qd, qe), g in zip(queries, got):
        orc = oracle.loop(frame_gap=1, sc_thr=KW["sc_distance_threshold"], icp_thr=KW["icp_fitness_threshold"],
                          max_candidates=KW["max_candidates"])
        for d, s in enumerate(streams):
            if d != qd:
                for c, f in zip(s.clouds, s.frames):
                    orc.add(c, f)
        orc.add(streams[qd].clouds[qe], Q_FRAME)
        want = orc.detect()
        assert [r["match_frame"] for r in g] == [r["match_frame"] for r in want]
        for rg, ro in zip(g, want):
            assert rg["scan_context_distance"] == ro["scan_context_distance"]
            assert abs(rg["icp_fitness"] - ro["icp_fitness"]) < 1e-6
            dT = rg["transform"] @ np.linalg.inv(ro["transform"])
            assert np.linalg.norm(dT[:3, 3]) < 1e-4 and rot_angle(dT[:3, :3]) < 1e-5
    assert any(len(g) > 0 for g in got)


@pytest.mark.gpu
def test_fleet_after_push_many(engine, synth, scene):
    """Four sessions on overlapping paths pushed together for 40 frames; then every session's scheduled entries are
    searched against the others.  Accepted transforms agree with the synth poses."""
    from conftest import rot_angle
    s = oracle_lib.small_sensor(16, 360)
    n_s, n_f = 4, 40
    # the same stretch of road, 0.5 m steps, each session 0.15 m further to the side; the node's threshold 0.2 keeps
    # the candidates to close revisits, which ICP from identity (loop_closure.hpp:99-109) resolves
    kw = dict(KW, sc_distance_threshold=0.2)
    pose = lambda k, i: (0.5 * i + 0.1 * k, 0.15 * k, 0.0)
    dets = [slam_b200.LoopClosureDetector(engine, frame_gap=50, **kw) for _ in range(n_s)]
    sess = [slam_b200.Odometry(engine, voxel=0.5, min_points=100, loop=d) for d in dets]
    held = [Stream([], []) for _ in range(n_s)]
    descs = [[] for _ in range(n_s)]
    truth = [[] for _ in range(n_s)]
    for i in range(n_f):
        frames = [synth.scan(s, scene, pose(k, i), 2000 + 50 * k + i) for k in range(n_s)]
        out = slam_b200.push_many(sess, frames, i, want_cloud=True, want_desc=True)
        for k, f in enumerate(out):
            if f.state != slam_b200.ODOM_SKIPPED:
                held[k].clouds.append(f.cloud)
                held[k].frames.append(i)
                descs[k].append(f.desc)
                truth[k].append(pose(k, i))
    for k in range(n_s):
        held[k].descs = np.stack(descs[k])
        assert dets[k].size() == len(held[k].clouds) > n_f // 2
    queries = [(k, e) for k in range(n_s) for e in range(0, dets[k].size(), 4)]
    lists, counts = slam_b200.candidates_across(dets, queries)
    got = slam_b200.detect_across(dets, queries)
    ref = reference(engine, held, queries, kw)
    n_acc = 0
    for i, (qd, qe) in enumerate(queries):
        d, db, ent, cnt, loops = ref[i]
        assert counts[i] == cnt and np.array_equal(lists[i][0], d)
        assert np.array_equal(lists[i][1], db) and np.array_equal(lists[i][2], ent)
        assert [r["match_frame"] for r in got[i]] == [r["match_frame"] for r in loops]
        for a, b in zip(got[i], loops):
            assert a["icp_fitness"] == b["icp_fitness"] and np.array_equal(a["transform"], b["transform"])
            assert a["scan_context_distance"] == b["scan_context_distance"]
            md = a["match_db"]
            me = held[md].frames.index(a["match_frame"])
            tq, tm = truth[qd][qe], truth[md][me]
            # ICP(query -> match) with the same heading: the query cloud moves by its offset from the match
            want = np.array([tq[0] - tm[0], tq[1] - tm[1], 0.0])
            assert np.linalg.norm(a["transform"][:3, 3] - want) < 0.2
            assert rot_angle(a["transform"][:3, :3]) < 0.02
            n_acc += 1
    assert n_acc > 0


@pytest.mark.gpu
def test_walk_past_the_short_list(engine, oracle, synth, scene):
    """More than 32 candidates over two detectors, the best 32 decoys that fail ICP, equal descriptors in both (ties go
    to the lower detector index), verify_chunk 3: acceptances come from rank >= 32 and equal the scratch detector's."""
    s = oracle_lib.small_sensor(16, 360)
    cloud = lambda p, seed: oracle.voxel_downsample(synth.scan(s, scene, p, seed), 0.5)[0]
    qc = cloud((0.0, 0.0, 0.0), 900)
    base = engine.sc_compute(qc)
    rng = np.random.default_rng(5)
    kw = dict(sc_distance_threshold=1e300, icp_fitness_threshold=0.3, max_candidates=2, verify_chunk=3)
    decoy = [base + rng.uniform(0, 0.01, 1200) * (base != 0) for _ in range(20)]
    streams = [Stream([qc], [0], base[None, :])]
    for d in (1, 2):
        clouds, descs = [], []
        for i in range(20):   # another place, 40 m away; detector 2 repeats detector 1's descriptors
            clouds.append(cloud((40.0 + 0.5 * (i % 4), 0.0, 0.0), 910 + 20 * d + i))
            descs.append(decoy[i])
        for i in range(2):    # the same place, with a descriptor further away
            clouds.append(cloud((0.3 * (i + 1) * d, 0.1, 0.0), 960 + 10 * d + i))
            descs.append(base + rng.uniform(0, 2.0, 1200) * (base != 0))
        streams.append(Stream(clouds, [1000 * d + i for i in range(len(clouds))], np.stack(descs)))
    dbs = [st.detector(engine, frame_gap=10, **kw) for st in streams]
    lists, counts, got = same_as_reference(engine, dbs, streams, [(0, 0)], kw, lambda f: f // 1000)
    assert counts[0] == 44
    d, db, ent = lists[0]
    assert all(d[j] == d[j + 1] and db[j] == 1 and db[j + 1] == 2 and ent[j] == ent[j + 1] for j in range(0, 32, 2))
    top = set(zip(db.tolist(), ent.tolist()))
    assert got[0] and all((r["match_db"], r["match_frame"] % 1000) not in top for r in got[0])


@pytest.mark.gpu
def test_edges(engine, streams):
    dbs = [s.detector(engine, frame_gap=50, **KW) for s in streams[:3]]
    empty = slam_b200.LoopClosureDetector(engine, frame_gap=50, **KW)
    before = [(d.size(), d.candidates_local(), d.detect()) for d in dbs]
    # empty detectors among the others, and a call whose only other detector is empty
    mixed = [dbs[0], empty, dbs[1], slam_b200.LoopClosureDetector(engine, frame_gap=5, **KW), dbs[2]]
    with_empty = streams[:1] + [Stream([], [])] + streams[1:2] + [Stream([], [])] + streams[2:3]
    # queries of three detectors in one tile of 8: a mixed pair mask
    queries = [(0, 20), (2, 3), (4, 15), (0, 2), (2, 20), (4, 0), (0, 10), (2, 12), (4, 5)]
    same_as_reference(engine, mixed, with_empty, queries, KW, lambda f: {0: 0, 1: 2, 2: 4}[f // 1000])
    lists, counts = slam_b200.candidates_across([dbs[0], empty], [(0, 3), (0, 20)])
    assert list(counts) == [0, 0] and all(len(x[0]) == 0 for x in lists)
    assert slam_b200.detect_across([dbs[0], empty], [(0, 3), (0, 20)]) == [[], []]
    assert slam_b200.detect_across([dbs[0]], [(0, 3)]) == [[]]
    # max_candidates = 0: no results
    kw0 = dict(KW, max_candidates=0)
    none = [s.detector(engine, frame_gap=50, **kw0) for s in streams[:2]]
    assert slam_b200.detect_across(none, [(0, 20), (1, 5)]) == [[], []]
    # the calls change no detector
    for d, (n, cand, det) in zip(dbs, before):
        assert d.size() == n
        assert all(np.array_equal(a, b) for a, b in zip(d.candidates_local(), cand))
        got = d.detect()
        assert [(r["match_frame"], r["icp_fitness"]) for r in got] == [(r["match_frame"], r["icp_fitness"]) for r in det]


@pytest.mark.gpu
def test_row_groups_match_the_one_query_search(engine):
    """Enough queries and columns that the distance matrix runs in several 32 MB groups (descriptor-only entries with
    tiny clouds): sampled rows equal the one-query search against each other detector, sorted by (distance, db, entry)."""
    rng = np.random.default_rng(11)
    sizes = (2100, 1500, 700)
    base = np.where(rng.uniform(size=(40, 60, 20)) < 0.35, rng.uniform(-1.7, 9.0, (40, 60, 20)), 0.0)

    def descs(n):
        d = base[rng.integers(0, 40, n)] + np.where(rng.uniform(size=(n, 60, 20)) < 0.05,
                                                    rng.normal(0, 0.5, (n, 60, 20)), 0.0)
        return np.stack([np.roll(x, int(s), axis=0) for x, s in zip(d, rng.integers(0, 60, n))]).reshape(n, -1)
    desc = [descs(n) for n in sizes]
    thr = float(np.median(engine.sc_distance_batch(desc[0][0], desc[1])))
    dbs = []
    for n, d in zip(sizes, desc):
        det = slam_b200.LoopClosureDetector(engine, frame_gap=5, sc_distance_threshold=thr)
        det.addFrames(rng.uniform(-20, 20, (n * 8, 3)), np.arange(n + 1) * 8, np.arange(n), d)
        dbs.append(det)
    queries = [(0, e) for e in range(sizes[0])] + [(2, e) for e in range(0, sizes[2], 3)]
    ld = sum((n + 7) // 8 * 8 for n in sizes)
    rows = (32 << 20) // (8 * ld) // 8 * 8
    assert len(queries) > 2 * rows   # at least three groups
    lists, counts = slam_b200.candidates_across(dbs, queries)
    sample = sorted({0, 1, rows - 1, rows, rows + 1, 2 * rows - 1, 2 * rows, len(queries) - 1} |
                    set(rng.integers(0, len(queries), 6).tolist()))
    for j in sample:
        qd, qe = queries[j]
        d = np.concatenate([engine.sc_distance_batch(desc[qd][qe], desc[o]) for o in range(3) if o != qd])
        db = np.concatenate([np.full(sizes[o], o) for o in range(3) if o != qd])
        e = np.concatenate([np.arange(sizes[o]) for o in range(3) if o != qd])
        keep = d < thr
        order = np.lexsort((e[keep], db[keep], d[keep]))
        assert counts[j] == keep.sum()
        assert np.array_equal(lists[j][0], d[keep][order][:32])
        assert np.array_equal(lists[j][1], db[keep][order][:32]) and np.array_equal(lists[j][2], e[keep][order][:32])


@pytest.mark.gpu
def test_argument_rules(engine, streams):
    a, b = (s.detector(engine, frame_gap=50, **KW) for s in streams[:2])
    other = slam_b200.Engine(0)
    try:
        foreign = streams[2].detector(other, frame_gap=50, **KW)
        w2 = slam_b200.LoopClosureDetector(engine, frame_gap=50, world=2, **KW)
        w2.addFrames(*streams[2].csr(), streams[2].frames)
        cases = [([a, b, foreign], [(0, 1)], "detector 2"),
                 ([a, b, a], [(0, 1)], "detector 2"),
                 ([a, w2], [(0, 1)], "detector 1"),
                 ([a, b], [(2, 1)], "query 0"),
                 ([a, b], [(0, 1), (1, -1)], "query 1"),
                 ([a, b], [(0, 1), (0, 2), (1, len(streams[1].clouds))], "query 2"),
                 ([a, b], [(-1, 0)], "query 0")]
        for field, value in [("sc_distance_threshold", 0.4), ("icp_fitness_threshold", 0.2), ("max_candidates", 2),
                             ("icp_max_iterations", 20), ("normals_k", 10), ("icp_tolerance", 1e-5),
                             ("verify_chunk", 4)]:
            det = slam_b200.LoopClosureDetector(engine, frame_gap=7, **KW)   # frame_gap may differ
            cfg = slam_b200.LoopConfigC.from_buffer_copy(det.cfg)
            setattr(cfg, field, value)
            h = slam_b200._P()
            engine._check(engine.lib.sb_loop_create(engine.h, C.byref(cfg), 0, 1, C.byref(h)))
            det.close()
            det.h, det.cfg = h, cfg
            det.addFrames(*streams[2].csr(), streams[2].frames)
            cases.append(([a, b, det], [(0, 1)], "detector 2: " + field))
        good = slam_b200.detect_across([a, b], [(0, 20)])
        for dbs, queries, msg in cases:
            for call in (slam_b200.detect_across, slam_b200.candidates_across):
                with pytest.raises(slam_b200.SlamB200Error) as ex:
                    call(dbs, queries)
                assert ex.value.status == 1 and msg in str(ex.value), str(ex.value)
                again = slam_b200.detect_across([a, b], [(0, 20)])   # a correct call right after
                assert [(r["match_frame"], r["icp_fitness"]) for r in again[0]] == \
                       [(r["match_frame"], r["icp_fitness"]) for r in good[0]]
    finally:
        other.close()


@pytest.mark.gpu
def test_search_launches_do_not_grow_with_detectors(engine):
    rng = np.random.default_rng(3)

    def launches(n_dbs):
        dbs = []
        for d in range(n_dbs):
            n = 40
            det = slam_b200.LoopClosureDetector(engine, frame_gap=5, sc_distance_threshold=0.3)
            det.addFrames(rng.uniform(-20, 20, (n * 8, 3)), np.arange(n + 1) * 8, np.arange(n),
                          rng.uniform(0, 3, (n, 1200)))
            dbs.append(det)
        queries = [(d, 3) for d in range(n_dbs)][:2]
        slam_b200.candidates_across(dbs, queries)   # warm
        c0 = engine.launch_count
        slam_b200.candidates_across(dbs, queries)
        return engine.launch_count - c0
    assert launches(2) == launches(16)
