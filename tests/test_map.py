"""Device-resident map (sb_map_*, slam_b200.Map, slam::b200::Map): the node's keyframe clouds, poses and occupancy cell
set kept on the device (slam_node.cpp:147-157, 177-238).  Every output is checked bit for bit against the stateless
entry points on the same clouds and poses (Engine.occupancy_cells / global_map[_f32] / transform_clouds_f32) and against
the oracle, after adds, pose updates, growth and failed calls.  The CPU tests model the cell table (open addressing,
insert limit at half load, doubling by rehash) and its growth rule.
"""
import ctypes as C
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "lidar-slam-from-scratch_b200", "python"))
import slam_b200  # noqa: E402

STREAM_RADIUS, STREAM_SCENE, STREAM_FRAMES = 10.5, 3, 78   # test_odom_session's loop-closure sequence
VOXEL = 0.5
WINDOW = 20                                               # slam_node.hpp:169: the last 20 world clouds
MASK64 = (1 << 64) - 1
GOLDEN = 0x9E3779B97F4A7C15
FIRST_ROWS, FIRST_ENTRIES, FIRST_TABLE_SLOTS = 1 << 20, 1024, 1 << 16   # map.cu


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


# ------------------------------------------------------------------ CPU: the ABI and the Python layer
def test_symbols_cover_every_map_entry_point():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "slam_b200.h")).read(), flags=re.S)
    declared = set(re.findall(r"\b(sb_map_[a-z0-9_]+)\s*\(", src)) | {"sb_odom_create2"}
    want = {"sb_map_create", "sb_map_free", "sb_map_reserve", "sb_map_size", "sb_map_rows", "sb_map_capacity",
            "sb_map_clear", "sb_map_add", "sb_map_set_poses", "sb_map_get_poses", "sb_map_occupancy_cells",
            "sb_map_world_f32", "sb_map_global", "sb_map_global_f32", "sb_odom_create2"}
    assert declared == want, declared ^ want
    assert want <= set(slam_b200.SYMBOLS)
    lib = slam_b200.load_library()
    for name in want:
        assert hasattr(lib, name), name
    assert slam_b200.ODOM_ADD_MAP == 4


def test_map_calls_refuse_null_handles():
    lib = slam_b200.load_library()
    h = C.c_void_p()
    assert lib.sb_map_create(None, None, C.byref(h)) == 1            # SB_ERR_INVALID_ARG
    assert lib.sb_map_add(None, None, 0, None) == 1
    assert lib.sb_map_set_poses(None, 0, 0, None) == 1
    assert lib.sb_map_occupancy_cells(None, None, 0, None) == 1
    assert lib.sb_map_global(None, 1.0, None, None) == 1
    assert lib.sb_map_size(None) == 0 and lib.sb_map_rows(None) == 0


class _FakeLib:
    """Answers sb_map_size / sb_map_rows; any other call means an argument check came too late."""

    def __init__(self, size):
        self.size = size

    def sb_map_size(self, h):
        return self.size

    def sb_map_rows(self, h):
        return 100 * self.size

    def __getattr__(self, name):
        raise AssertionError(f"{name} reached the library with bad arguments")


def fake_map(size):
    m = slam_b200.Map.__new__(slam_b200.Map)

    class E:
        h = C.c_void_p(1)
        lib = _FakeLib(size)

        def _check(self, s):
            raise AssertionError("no call expected")

    m.e, m.h = E(), C.c_void_p(1)
    return m


def test_python_argument_checks_reject_bad_input_before_any_call():
    m = fake_map(5)
    with pytest.raises(ValueError):
        m.add(np.zeros((4, 3)), np.eye(3))                     # a pose is 4x4
    with pytest.raises(ValueError):
        m.add(np.zeros((4, 2)), np.eye(4))                     # rows are xyz
    with pytest.raises(ValueError):
        m.set_poses(np.zeros((2, 4, 3)))
    with pytest.raises(ValueError):
        m.set_poses(np.tile(np.eye(4), (3, 1, 1)), first=3)    # entries 3..5 of 5
    with pytest.raises(ValueError):
        m.set_poses(np.eye(4), first=-1)
    with pytest.raises(ValueError):
        m.poses(4, 2)
    with pytest.raises(ValueError):
        m.world_f32(0, 6)
    with pytest.raises(ValueError):
        m.world_f32(-1, 1)
    with pytest.raises(ValueError):
        m.occupancy_cells(capacity=-1)
    m.h = None   # close() of a map whose engine is gone drops the handle
    m.e.h = None
    m.close()


# ------------------------------------------------------------------ CPU: model of map.cu's cell table
def cell_key(x, y):
    """occ_key's packing: biased x in the high word, biased y in the low word."""
    return (((x ^ 0x80000000) & 0xffffffff) << 32) | ((y ^ 0x80000000) & 0xffffffff)


class TableModel:
    """map.cu's set of cell keys: linear probing from (key * golden) >> (64 - log2 slots), ~0 = empty.  A launch claims
    at most `limit` slots (table_insert); a launch that needs more flags FULL, the table doubles by rehash
    (k_map_rehash) and the launch's keys go in again.  Lanes of a warp with equal keys probe once (__match_any_sync)."""

    EMPTY = MASK64

    def __init__(self, slots):
        self.slots = [self.EMPTY] * slots
        self.n = 0
        self.max_probe = 0
        self.growths = 0

    def _slot(self, key):
        return ((key * GOLDEN) & MASK64) >> (64 - (len(self.slots).bit_length() - 1))

    def _insert(self, key, count, limit):
        mask = len(self.slots) - 1
        s = self._slot(key)
        for step in range(len(self.slots)):
            cur = self.slots[s]
            if cur == key:
                return count, False
            if cur == self.EMPTY:
                if count >= limit:
                    return count, True
                self.slots[s] = key
                self.max_probe = max(self.max_probe, step + 1)
                return count + 1, False
            s = (s + 1) & mask
        return count, True

    def _resize(self, slots):
        old = [k for k in self.slots if k != self.EMPTY]
        self.slots = [self.EMPTY] * slots
        for k in old:
            self._insert(k, 0, 1 << 62)
        self.growths += 1

    def launch(self, keys, rng):
        """One k_map_occ_insert launch over `keys` (a row each) in a random warp order; returns (count, full)."""
        keys = list(keys)
        warps = [keys[i:i + 32] for i in range(0, len(keys), 32)]
        order = rng.permutation(len(warps))
        limit = len(self.slots) // 2 - self.n
        count, full = 0, False
        for w in order:
            for lane, k in enumerate(warps[w]):
                if k == self.EMPTY or k in warps[w][:lane]:
                    continue                     # filtered out, or not the lowest lane of its key in the warp
                count, f = self._insert(k, count, limit)
                full |= f
        return count, full

    def add(self, keys, rng):
        """map_add_finish: relaunch after each doubling, then keep the load at most one half."""
        inserted, full = self.launch(keys, rng)
        while full:
            self.n += inserted
            self._resize(2 * len(self.slots))
            c, full = self.launch(keys, rng)
            inserted = c
        self.n += inserted
        while 2 * self.n > len(self.slots):
            self._resize(2 * len(self.slots))

    def cells(self):
        """Extraction: the occupied slots compacted and sorted (unsigned key order), unpacked."""
        keys = np.array(sorted(k for k in self.slots if k != self.EMPTY), dtype=np.uint64)
        x = ((keys >> np.uint64(32)).astype(np.uint32) ^ np.uint32(0x80000000)).view(np.int32)
        y = ((keys & np.uint64(0xffffffff)).astype(np.uint32) ^ np.uint32(0x80000000)).view(np.int32)
        return np.stack([x, y], axis=1) if len(keys) else np.zeros((0, 2), dtype=np.int32)


def test_cell_table_model_gives_the_set_np_unique_gives():
    rng = np.random.default_rng(11)
    T = TableModel(16)
    rows = []
    for call in range(12):
        n = int(rng.integers(20, 400))
        # runs of equal cells as neighbouring rows of a scan give them, some rows filtered out
        xy = np.repeat(rng.integers(-60, 60, size=(n // 4 + 1, 2)), 4, axis=0)[:n]
        keys = [cell_key(int(x), int(y)) for x, y in xy]
        drop = rng.random(n) < 0.1
        keys = [TableModel.EMPTY if d else k for k, d in zip(keys, drop)]
        rows.extend(xy[~drop].tolist())
        T.add(keys, rng)
        want = np.unique(np.array(rows, dtype=np.int32).reshape(-1, 2), axis=0)   # lexicographic (x, y)
        got = T.cells()
        assert np.array_equal(got, want), call
        assert T.n == len(want) and 2 * T.n <= len(T.slots), call
    assert T.growths >= 4 and T.max_probe > 1      # the table grew inside calls, and keys collided


def test_unsigned_key_order_is_the_signed_cell_order():
    rng = np.random.default_rng(2)
    xy = rng.integers(-2**31 + 1, 2**31 - 1, size=(2000, 2))
    xy[:20] = [[0, 0], [-1, 0], [0, -1], [-1, -1], [1, -1], [-2**31 + 1, 5], [2**31 - 2, -5], [3, 2**31 - 2],
               [3, -2**31 + 1], [-7, 7], [7, -7], [0, 1], [1, 0], [-1, 1], [5, 5], [5, 4], [4, 5], [-5, -5], [-5, -4],
               [-4, -5]]
    keys = [cell_key(int(x), int(y)) for x, y in xy]
    by_key = [tuple(v) for v in xy[np.argsort(np.array(keys, dtype=np.uint64), kind="stable")]]
    assert by_key == sorted(tuple(v) for v in xy.tolist())


def doubled(cap, need, first):
    c = cap if cap > 0 else max(first, 1)
    while c < need:
        c *= 2
    return c


def capacity_model(adds, reserve=None):
    """map.cu's growth rule: (entries, rows, table slots) after each add of (rows, cells after the add)."""
    if reserve is None:
        caps = [FIRST_ENTRIES, 0, FIRST_TABLE_SLOTS]
    else:
        e, r, c = reserve
        caps = [max(FIRST_ENTRIES, e), r if r > 0 else 0, doubled(FIRST_TABLE_SLOTS, 2 * c, 1)]
    out, entries, rows = [], 0, 0
    for n, cells in adds:
        entries, rows = entries + 1, rows + n
        if entries > caps[0]:
            caps[0] = doubled(caps[0], entries, FIRST_ENTRIES)
        if rows > caps[1]:
            caps[1] = doubled(caps[1], rows, FIRST_ROWS)
        if 2 * cells > caps[2]:
            caps[2] = doubled(caps[2], 2 * cells, FIRST_TABLE_SLOTS)
        out.append(tuple(caps))
    return out


def test_capacity_model():
    caps = capacity_model([(600000, 20000), (600000, 40000), (0, 40000), (2000000, 500000)])
    assert caps == [(1024, 1 << 20, 1 << 16), (1024, 1 << 21, 1 << 17), (1024, 1 << 21, 1 << 17),
                    (1024, 1 << 22, 1 << 20)]
    assert capacity_model([(600000, 20000)] * 3, reserve=(10, 1 << 22, 100000)) == [(1024, 1 << 22, 1 << 18)] * 3


def test_mirror_map_compiles_in_both_dense_branches():
    prog = r'''
#include "slam_viz/core/map.hpp"
#include "slam_viz/core/odometry.hpp"
int main() {
    slam::b200::Map map;
    slam::PointCloud::Matrix rows(2, 3);
    map.add(rows, slam::Transformation::identity());
    map.setPoses(map.poses(), 0);
    slam::b200::Odometry odom(slam::b200::OdometryConfig(), nullptr, &map);
    return (int)(map.occupancyCells().size() + map.worldF32(0, 1).size() + map.globalMap(1.0).size() +
                 map.globalMapF32(1.0).size());
}
'''
    host = os.path.join(ROOT, "lidar-slam-from-scratch_b200", "host")
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "m.cpp")
        with open(src, "w") as fh:
            fh.write(prog)
        for extra in ([], ["-I" + os.path.join(ROOT, "oracle", "eigen_standin")]):
            subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wno-unused-function", *extra,
                                   "-I" + os.path.join(ROOT, "include"), "-I" + host, "-c", src, "-o",
                                   os.path.join(d, "m.o")])


# ------------------------------------------------------------------ GPU fixtures
def cores():
    return os.cpu_count() or 1


@pytest.fixture(scope="module")
def stream(synth):
    sys.path.insert(0, ROOT)
    import bench
    world = synth.scene(STREAM_SCENE, n_boxes=400, path_kind=1, radius=STREAM_RADIUS)
    return [synth.scan(bench.SENSOR, world, synth.pose(1, STREAM_RADIUS, float(i)), 500 + i, threads=cores())
            for i in range(STREAM_FRAMES)]


@pytest.fixture(scope="module")
def keyframes(engine, stream):
    """The session's downsampled clouds and poses of the stream: what the node keeps as downsampled_clouds_ / poses_."""
    odom = slam_b200.Odometry(engine)
    frames = [odom.push(s, i, want_cloud=True) for i, s in enumerate(stream)]
    odom.close()
    return [f.cloud for f in frames], np.stack([f.pose for f in frames])


def csr(clouds):
    off = np.r_[0, np.cumsum([len(c) for c in clouds])].astype(np.int64)
    pts = np.concatenate(clouds) if clouds else np.zeros((0, 3))
    return pts, off


def stateless(engine, clouds, poses, window=WINDOW, voxel=2 * VOXEL, grid=None):
    pts, off = csr(clouds)
    Ts = np.asarray(poses).reshape(-1, 4, 4)
    k = max(len(clouds) - window, 0)
    wpts, woff = csr(clouds[k:])
    return dict(cells=engine.occupancy_cells(pts, off, Ts, **(grid or {})), gm=engine.global_map(pts, off, Ts, voxel),
                gm32=engine.global_map_f32(pts, off, Ts, voxel),
                win=engine.transform_clouds_f32(wpts, woff, Ts[k:]) if len(wpts) else np.zeros((0, 3), np.float32))


def assert_map_equals(m, want, window=WINDOW, voxel=2 * VOXEL, what=""):
    cells, count = m.occupancy_cells()
    assert count == want["cells"][1] and same_bits(cells, want["cells"][0]), what
    assert same_bits(m.global_map(voxel), want["gm"]), what
    assert same_bits(m.global_map(voxel, f32=True), want["gm32"]), what
    k = max(len(m) - window, 0)
    assert same_bits(m.world_f32(k, len(m) - k), want["win"]), what


def perturbed(poses, seed, scale=1.0):
    """A loop-closure style correction: every pose moved by a small rigid motion that grows along the sequence."""
    rng = np.random.default_rng(seed)
    out = []
    for i, P in enumerate(poses):
        a = scale * 0.002 * i * rng.uniform(0.5, 1.0)
        D = np.eye(4)
        D[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
        D[:3, 3] = scale * 0.01 * i * rng.uniform(-1, 1, 3)
        out.append(D @ P)
    return np.stack(out)


# ------------------------------------------------------------------ 1. entry by entry
@pytest.mark.gpu
def test_every_add_matches_the_stateless_calls_and_the_oracle(engine, oracle, keyframes):
    clouds, poses = keyframes
    m = slam_b200.Map(engine)
    for i, (c, P) in enumerate(zip(clouds, poses)):
        m.add(c, P)
        assert len(m) == i + 1 and m.rows == sum(len(x) for x in clouds[:i + 1])
        want = stateless(engine, clouds[:i + 1], poses[:i + 1])
        assert_map_equals(m, want, what=i)
        pts, off = csr(clouds[:i + 1])
        ref = oracle.occupancy_cells(pts, off, poses[:i + 1])
        assert np.array_equal(m.occupancy_cells()[0], ref), i
        if i % 10 == 0 or i == len(clouds) - 1:
            world = np.concatenate([oracle.transform_cloud(x, T) for x, T in zip(clouds[:i + 1], poses[:i + 1])])
            ref_gm, _ = oracle.voxel_downsample(world, 2 * VOXEL)
            assert same_bits(m.global_map(2 * VOXEL), ref_gm), i
            assert same_bits(m.global_map(2 * VOXEL, f32=True), ref_gm.astype(np.float32)), i
    assert same_bits(m.poses(), poses)
    assert same_bits(m.global_map(0.0), np.concatenate([oracle.transform_cloud(x, T) for x, T in zip(clouds, poses)]))
    print(f"[map] {len(m)} entries, {m.rows} rows, {m.occupancy_cells()[1]} cells: every add equal to the stateless "
          f"calls and the oracle")
    m.close()


# ------------------------------------------------------------------ 2. pose updates
@pytest.mark.gpu
def test_set_poses_rebuilds_what_the_stateless_calls_give(engine, oracle, keyframes):
    clouds, poses = keyframes
    m = slam_b200.Map(engine)
    for c, P in zip(clouds, poses):
        m.add(c, P)
    before = set(map(tuple, m.occupancy_cells()[0].tolist()))
    new = perturbed(poses, 1)
    m.set_poses(new)                                     # a correction of every entry
    assert same_bits(m.poses(), new)
    assert_map_equals(m, stateless(engine, clouds, new), what="all")
    pts, off = csr(clouds)
    assert np.array_equal(m.occupancy_cells()[0], oracle.occupancy_cells(pts, off, new))
    sub = perturbed(new[30:55], 2, scale=3.0)            # a sub-range
    m.set_poses(sub, first=30)
    both = new.copy()
    both[30:55] = sub
    assert same_bits(m.poses(), both) and same_bits(m.poses(30, 25), sub)
    assert_map_equals(m, stateless(engine, clouds, both), what="sub-range")
    # entries moved 500 m away: their old cells go, and their rows leave max_range of nothing else
    far = both.copy()
    far[:, 0, 3] += np.where(np.arange(len(far)) < 40, 500.0, 0.0)
    m.set_poses(far)
    after = set(map(tuple, m.occupancy_cells()[0].tolist()))
    assert before - after
    assert_map_equals(m, stateless(engine, clouds, far), what="far")
    m.close()


# ------------------------------------------------------------------ 3. the session feeding the map
@pytest.mark.gpu
def test_session_with_add_map_leaves_the_map_sb_map_add_builds(engine, stream):
    scans = list(stream[:40])
    for k in (10, 25):                                   # below min_points: skipped, the pose repeats
        scans.insert(k, stream[k][::200].copy())
    det_a, det_b = slam_b200.LoopClosureDetector(engine), slam_b200.LoopClosureDetector(engine)
    m = slam_b200.Map(engine)
    with_map = slam_b200.Odometry(engine, loop=det_a, map=m)
    plain = slam_b200.Odometry(engine, loop=det_b)
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_odom_session import frame_bits
    got, ref = [], []
    for i, s in enumerate(scans):
        got.append(with_map.push(s, i, detect=(i == 45), want_cloud=True, want_world_f32=True, want_desc=True))
        ref.append(plain.push(s, i, detect=(i == 45), want_cloud=True, want_world_f32=True, want_desc=True))
        assert same_bits(frame_bits(got[-1]), frame_bits(ref[-1])), i
    skipped = [i for i, f in enumerate(got) if f.state == slam_b200.ODOM_SKIPPED]
    assert skipped == [10, 25]
    with_map.close()
    plain.close()
    clouds = [np.zeros((0, 3)) if f.state == slam_b200.ODOM_SKIPPED else f.cloud for f in got]
    poses = np.stack([f.pose for f in got])
    assert len(m) == len(scans) and same_bits(m.poses(), poses) and m.rows == sum(len(c) for c in clouds)
    built = slam_b200.Map(engine)
    for c, P in zip(clouds, poses):
        built.add(c, P)
    want = stateless(engine, clouds, poses)
    assert_map_equals(m, want, what="session")
    assert_map_equals(built, want, what="sb_map_add")
    for i in range(len(m)):   # the window of every frame: its own world_f32
        if i not in skipped:
            assert same_bits(m.world_f32(i, 1), got[i].world_f32), i
        else:
            assert m.world_f32(i, 1).shape == (0, 3)
    for x in (m, built, det_a, det_b):
        x.close()


# ------------------------------------------------------------------ 4. growth
@pytest.mark.gpu
def test_growth_without_reserve_and_no_growth_with_it(engine, synth, scene):
    sys.path.insert(0, ROOT)
    import bench
    # raw scans (~100 k rows each) as entries, every row of them a cell (no height or range filter): the row pool and the
    # cell table double several times
    grid = dict(height_min=-1e9, height_max=1e9, max_range=1e9)
    raws = [synth.scan(bench.SENSOR, scene, (1.5 * i, 0.2 * i, 0.03 * i), 700 + i, threads=cores()) for i in range(24)]
    poses = []
    for i in range(len(raws)):
        P = np.eye(4)
        a = 0.05 * i
        P[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
        P[:3, 3] = [40.0 * i, -25.0 * i, 0.1]
        poses.append(P)
    m = slam_b200.Map(engine, **grid)
    assert m.capacity() == (FIRST_ENTRIES, 0, FIRST_TABLE_SLOTS)
    counts, caps = [], []
    for i, (c, P) in enumerate(zip(raws, poses)):
        m.add(c, P)
        counts.append(m.occupancy_cells(capacity=0)[1])
        caps.append(m.capacity())
        if i in (0, 7, 15):
            assert_map_equals(m, stateless(engine, raws[:i + 1], poses[:i + 1], grid=grid), what=i)
    want = stateless(engine, raws, poses, grid=grid)
    assert_map_equals(m, want, what="grown")
    model = capacity_model([(len(c), n) for c, n in zip(raws, counts)])
    assert caps == model
    rows_growths = len({c[1] for c in caps}) - 1
    table_growths = len({c[2] for c in caps} | {FIRST_TABLE_SLOTS}) - 1
    assert rows_growths >= 2 and table_growths >= 3, caps
    # reserve up front: no buffer grows on any add, the same bits
    r = slam_b200.Map(engine, **grid)
    r.reserve(len(raws), sum(len(c) for c in raws), counts[-1])
    c0 = r.capacity()
    for c, P in zip(raws, poses):
        r.add(c, P)
        assert r.capacity() == c0
    assert capacity_model([(len(c), n) for c, n in zip(raws, counts)],
                          reserve=(len(raws), sum(len(c) for c in raws), counts[-1]))[-1] == c0
    assert_map_equals(r, want, what="reserved")
    # every entry first at one pose (few cells), then spread out by set_poses: the table grows inside the rebuild
    g = slam_b200.Map(engine, **grid)
    for c in raws:
        g.add(c, poses[0])
    before = g.capacity()[2]
    g.set_poses(np.stack(poses))
    assert g.capacity()[2] > before and g.occupancy_cells(capacity=0)[1] == counts[-1]
    assert_map_equals(g, want, what="rebuild")
    g.close()
    print(f"[map] growth: capacities {caps[0]} -> {caps[-1]} ({rows_growths} row-pool and {table_growths} table "
          f"doublings), {counts[-1]} cells")
    m.close()
    r.close()


# ------------------------------------------------------------------ 5. failures and edge cases
@pytest.mark.gpu
def test_failed_calls_leave_the_map_unchanged(engine, keyframes, stream):
    clouds, poses = keyframes
    m = slam_b200.Map(engine)
    for c, P in zip(clouds[:30], poses[:30]):
        m.add(c, P)

    def state():
        return (len(m), m.rows, m.occupancy_cells(), m.poses(), m.global_map(2 * VOXEL), m.world_f32(10, 20))

    def same_state(a, b):
        return (a[0], a[1], a[2][1]) == (b[0], b[1], b[2][1]) and all(
            same_bits(x, y) for x, y in ((a[2][0], b[2][0]), (a[3], b[3]), (a[4], b[4]), (a[5], b[5])))

    s0 = state()
    bad = clouds[30].copy()
    bad[len(bad) // 2, 1] = np.nan
    for cloud, pose in ((bad, poses[30]), (clouds[30], np.full((4, 4), np.inf))):
        with pytest.raises(slam_b200.SlamB200Error) as e:
            m.add(cloud, pose)
        assert e.value.status == 5 and same_state(state(), s0)
    bad_poses = poses[:30].copy()
    bad_poses[7, 1, 3] = np.nan
    far = poses[:30].copy()
    far[3, 0, 3] = 1e12                                   # cells beyond int: SB_ERR_RANGE as k_occ_keys gives it
    for P in (bad_poses, far):
        with pytest.raises(slam_b200.SlamB200Error) as e:
            m.set_poses(P)
        assert e.value.status == 5 and same_state(state(), s0)
    with pytest.raises(slam_b200.SlamB200Error) as e:
        engine.occupancy_cells(*csr(clouds[:30]), far)
    assert e.value.status == 5
    # a push that fails (non-finite row) leaves the map it feeds unchanged; the next push adds normally
    odom = slam_b200.Odometry(engine, map=m)
    raw = stream[30].copy()
    raw[5, 0] = np.inf
    with pytest.raises(slam_b200.SlamB200Error):
        odom.push(raw, 30)
    assert same_state(state(), s0)
    odom.close()
    # the rows of a failed add are overwritten by the next one
    m.add(clouds[30], poses[30])
    assert_map_equals(m, stateless(engine, clouds[:31], poses[:31]), what="after failures")
    # capacity smaller than the count: the first cells and the full count
    cells, count = m.occupancy_cells()
    part, c2 = m.occupancy_cells(capacity=17)
    assert c2 == count > 17 and np.array_equal(part, cells[:17])
    assert m.occupancy_cells(capacity=0)[0].shape == (0, 2)
    # empty map and empty entries
    m.clear()
    cells, count = m.occupancy_cells()
    assert len(m) == 0 and m.rows == 0 and count == 0 and cells.shape == (0, 2)
    assert m.global_map(2 * VOXEL).shape == (0, 3) and m.global_map(1.0, f32=True).shape == (0, 3)
    assert m.world_f32(0, 0).shape == (0, 3)
    m.add(np.zeros((0, 3)), poses[0])
    assert len(m) == 1 and m.occupancy_cells()[1] == 0 and m.world_f32(0, 1).shape == (0, 3)
    m.add(clouds[0], poses[0])
    assert_map_equals(m, stateless(engine, [np.zeros((0, 3)), clouds[0]], poses[[0, 0]]), what="after clear")
    m.close()


# ------------------------------------------------------------------ 6. scale
@pytest.mark.gpu
def test_two_thousand_entries_match_sb_occupancy_cells(engine, keyframes):
    clouds, poses = keyframes
    n = 2000
    cl = [clouds[i % len(clouds)] for i in range(n)]
    Ts = []
    for i in range(n):   # the stream's clouds laid along a 4 km path: every entry its own place
        P = poses[i % len(poses)].copy()
        a = 2 * np.pi * i / n
        R = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])
        P[:3, :3] = R @ P[:3, :3]
        P[:3, 3] = R @ P[:3, 3] + [640.0 * np.cos(a), 640.0 * np.sin(a), 0.0]
        Ts.append(P)
    Ts = np.stack(Ts)
    m = slam_b200.Map(engine)
    for c, P in zip(cl, Ts):
        m.add(c, P)
    pts, off = csr(cl)
    assert m.rows == len(pts) > 8_000_000
    cells, count = m.occupancy_cells()
    ref, rc = engine.occupancy_cells(pts, off, Ts)
    assert count == rc and np.array_equal(cells, ref)
    new = perturbed(Ts, 5, scale=0.1)
    m.set_poses(new)
    cells, count = m.occupancy_cells()
    ref, rc = engine.occupancy_cells(pts, off, new)
    assert count == rc and np.array_equal(cells, ref)
    assert same_bits(m.world_f32(n - WINDOW, WINDOW), engine.transform_clouds_f32(*csr(cl[-WINDOW:]), new[-WINDOW:]))
    print(f"[map] {n} entries, {m.rows} rows: {count} cells equal to sb_occupancy_cells, before and after set_poses")
    m.close()
