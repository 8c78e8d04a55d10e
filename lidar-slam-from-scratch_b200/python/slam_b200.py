"""ctypes host layer over libslam_b200.so (include/slam_b200.h).

The reference's hot path is a header-only C++ API (slam_viz/include/slam_viz/core/*.hpp); this module gives the same
names and argument meaning to Python callers (tests, bench.py) on top of the C ABI:

    voxel_downsample(points, voxel)            file_utils.hpp:41-44
    KDTree(points).nearest_batch / k_nearest   kdtree.hpp:18-186
    estimate_normals(points, tree, k)          icp.hpp:23-67
    solve_point_to_plane(src, tgt, normals)    icp.hpp:89-144
    icp_point_to_plane(source, target, cfg)    icp.hpp:157-258
    ScanContext(cloud).distance(other)         scan_context.hpp:24-145
    LoopClosureDetector(cfg).addFrame/detect   loop_closure.hpp:41-149
    LoopClosureDetector.addFrames/detect_batch the same over a whole recorded sequence (slam_node.cpp:159-167)
    Odometry(engine).push(scan, i)             SlamNode::process_frame one scan per call (slam_node.cpp:118-175)
    push_many(sessions, scans, frame_idx)      one scan into each of many sessions in one call (many streams, one GPU)
    Map(engine).add / set_poses / ...          the node's keyframe clouds, poses and occupancy grid on the device

There is no CPU implementation here: if the shared library is missing, or no sm_100 device is usable, construction
fails loudly.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# SB_LIB_PATH: another build of the same library (A/B measurements of two builds in one job)
_LIB_PATH = os.environ.get("SB_LIB_PATH") or os.path.join(os.path.dirname(_HERE), "libslam_b200.so")

SB_SC_SIZE = 1200
SB_MAX_K = 32
SB_MAX_ICP_ITERATIONS = 128
SB_LOOP_SELECT_MAX = 32

STATUS = {0: "SB_OK", 1: "SB_ERR_INVALID_ARG", 2: "SB_ERR_EMPTY", 3: "SB_ERR_CUDA", 4: "SB_ERR_NO_DEVICE",
          5: "SB_ERR_RANGE", 6: "SB_ERR_CAPACITY"}


class SlamB200Error(RuntimeError):
    def __init__(self, status, msg=""):
        super().__init__(f"{STATUS.get(status, status)}: {msg}")
        self.status = status


class ICPConfigC(C.Structure):
    _fields_ = [("max_iterations", C.c_int32), ("normals_k", C.c_int32), ("tolerance", C.c_double),
                ("min_error", C.c_double), ("initial_transform", C.c_double * 16)]


class ICPResultC(C.Structure):
    _fields_ = [("transformation", C.c_double * 16), ("final_error", C.c_double), ("converged", C.c_int32),
                ("num_iterations", C.c_int32), ("history_len", C.c_int32), ("status", C.c_int32),
                ("error_history", C.c_double * (SB_MAX_ICP_ITERATIONS + 1))]


class LoopConfigC(C.Structure):
    _fields_ = [("frame_gap", C.c_int32), ("max_candidates", C.c_int32), ("sc_distance_threshold", C.c_double),
                ("icp_fitness_threshold", C.c_double), ("icp_max_iterations", C.c_int32), ("normals_k", C.c_int32),
                ("icp_tolerance", C.c_double), ("verify_chunk", C.c_int32), ("reserved", C.c_int32)]


class LoopResultC(C.Structure):
    _fields_ = [("query_frame", C.c_int32), ("match_frame", C.c_int32), ("transform", C.c_double * 16),
                ("scan_context_distance", C.c_double), ("icp_fitness", C.c_double)]


class PoseFactorC(C.Structure):
    _fields_ = [("kind", C.c_int32), ("from_", C.c_int32), ("to", C.c_int32), ("pad", C.c_int32),
                ("relative", C.c_double * 16), ("fitness", C.c_double), ("noise_scale", C.c_double)]


class OdomConfigC(C.Structure):
    _fields_ = [("voxel", C.c_double), ("min_points", C.c_int32), ("reserved", C.c_int32), ("max_error", C.c_double),
                ("icp", ICPConfigC), ("initial_pose", C.c_double * 16)]


class OdomFrameC(C.Structure):
    _fields_ = [("frame_idx", C.c_int32), ("state", C.c_int32), ("n_points", C.c_int64), ("pose", C.c_double * 16),
                ("icp", ICPResultC), ("n_loops", C.c_int32), ("pad", C.c_int32)]


ODOM_ADD_FRAME, ODOM_DETECT, ODOM_ADD_MAP = 1, 2, 4
ODOM_FIRST, ODOM_REGISTERED, ODOM_SKIPPED = 0, 1, 2


FACTOR_DTYPE = np.dtype([("kind", "<i4"), ("from", "<i4"), ("to", "<i4"), ("pad", "<i4"), ("relative", "<f8", (4, 4)),
                         ("fitness", "<f8"), ("noise_scale", "<f8")])

_P = C.c_void_p
_D = C.POINTER(C.c_double)
_I32 = C.POINTER(C.c_int32)
_I64 = C.POINTER(C.c_int64)

# every symbol include/slam_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "sb_version": (C.c_char_p, []),
    "sb_ctx_create": (C.c_int, [C.c_int, _P, C.POINTER(_P)]),
    "sb_ctx_destroy": (None, [_P]),
    "sb_last_error": (C.c_char_p, [_P]),
    "sb_ctx_synchronize": (C.c_int, [_P]),
    "sb_ctx_launch_count": (C.c_int64, [_P]),
    "sb_ctx_set_profiling": (C.c_int, [_P, C.c_int]),
    "sb_ctx_stage_ms": (C.c_int, [_P, _D]),
    "sb_ctx_stage_host_ms": (C.c_int, [_P, _D]),
    "sb_ctx_last_counts": (C.c_int, [_P, _I64]),
    "sb_ctx_last_voxel_path": (C.c_int, [_P]),
    "sb_default_icp_config": (None, [C.POINTER(ICPConfigC)]),
    "sb_default_loop_config": (None, [C.POINTER(LoopConfigC)]),
    "sb_voxel_downsample": (C.c_int, [_P, _D, C.c_int64, C.c_double, _D, _I64, _I64]),
    "sb_voxel_downsample_batch": (C.c_int, [_P, _D, _I64, C.c_int32, C.c_double, _D, _I64, _I64]),
    "sb_voxel_downsample_batch_dev": (C.c_int, [_P, _P, _I64, C.c_int32, C.c_double, _P, _I64, _P]),
    "sb_index_build": (C.c_int, [_P, _D, C.c_int64, C.POINTER(_P)]),
    "sb_index_free": (None, [_P]),
    "sb_index_size": (C.c_int64, [_P]),
    "sb_index_nearest_batch": (C.c_int, [_P, _D, C.c_int64, _I32, _D]),
    "sb_index_knn": (C.c_int, [_P, _D, C.c_int64, C.c_int32, _I32, _D]),
    "sb_index_find_correspondences": (C.c_int, [_P, _D, C.c_int64, _D, _D]),
    "sb_estimate_normals": (C.c_int, [_P, C.c_int32, _D, _D]),
    "sb_solve_point_to_plane": (C.c_int, [_P, _D, _D, _D, C.c_int64, _D]),
    "sb_icp_point_to_plane": (C.c_int, [_P, _D, C.c_int64, _D, C.c_int64, C.POINTER(ICPConfigC), C.POINTER(ICPResultC)]),
    "sb_register_batch": (C.c_int, [_P, _D, _I64, C.c_int32, C.c_double, _I32, _I32, C.c_int32,
                                    C.POINTER(ICPConfigC), C.POINTER(ICPResultC), _D]),
    "sb_register_batch_dev": (C.c_int, [_P, _P, _I64, C.c_int32, C.c_double, _I32, _I32, C.c_int32,
                                        C.POINTER(ICPConfigC), C.POINTER(ICPResultC), _D]),
    "sb_register_batch_f32": (C.c_int, [_P, _P, C.c_int32, _I64, C.c_int32, C.c_double, _I32, _I32, C.c_int32,
                                        C.POINTER(ICPConfigC), C.POINTER(ICPResultC), _D]),
    "sb_register_batch_f32_dev": (C.c_int, [_P, _P, C.c_int32, _I64, C.c_int32, C.c_double, _I32, _I32, C.c_int32,
                                            C.POINTER(ICPConfigC), C.POINTER(ICPResultC), _D]),
    "sb_voxel_downsample_batch_f32": (C.c_int, [_P, _P, C.c_int32, _I64, C.c_int32, C.c_double, _D, _I64, _I64]),
    "sb_sc_compute": (C.c_int, [_P, _D, C.c_int64, _D]),
    "sb_sc_distance": (C.c_int, [_P, _D, _D, _D]),
    "sb_sc_distance_batch": (C.c_int, [_P, _D, _D, C.c_int32, _D]),
    "sb_sc_keys": (C.c_int, [_P, _D, _D, _D]),
    "sb_loop_create": (C.c_int, [_P, C.POINTER(LoopConfigC), C.c_int32, C.c_int32, C.POINTER(_P)]),
    "sb_loop_free": (None, [_P]),
    "sb_loop_reserve": (C.c_int, [_P, C.c_int64, C.c_int64]),
    "sb_loop_add_frame": (C.c_int, [_P, _D, C.c_int64, C.c_int32]),
    "sb_loop_add_frame_desc": (C.c_int, [_P, _D, C.c_int64, C.c_int32, _D]),
    "sb_loop_size": (C.c_int64, [_P]),
    "sb_loop_clear": (C.c_int, [_P]),
    "sb_loop_detect": (C.c_int, [_P, C.POINTER(LoopResultC), C.c_int32, _I32]),
    "sb_loop_candidates_local": (C.c_int, [_P, _D, _I32, C.c_int32, _I32]),
    "sb_loop_verify_entries": (C.c_int, [_P, _I32, _D, C.c_int32, C.POINTER(LoopResultC), _I32]),
    "sb_loop_add_frames": (C.c_int, [_P, _D, _I64, C.c_int32, _I32, _D]),
    "sb_loop_candidates_batch": (C.c_int, [_P, _I32, C.c_int32, C.c_int32, _D, _I32, _I32]),
    "sb_loop_detect_batch": (C.c_int, [_P, _I32, C.c_int32, C.POINTER(LoopResultC), _I32]),
    "sb_loop_candidates_across": (C.c_int, [C.POINTER(_P), C.c_int32, _I32, _I32, C.c_int32, C.c_int32, _D, _I32, _I32,
                                            _I32]),
    "sb_loop_detect_across": (C.c_int, [C.POINTER(_P), C.c_int32, _I32, _I32, C.c_int32, C.POINTER(LoopResultC), _I32,
                                        _I32]),
    "sb_odometry_poses": (C.c_int, [_P, C.POINTER(ICPResultC), C.c_int32, C.c_double, _D, _D]),
    "sb_default_odom_config": (None, [C.POINTER(OdomConfigC)]),
    "sb_odom_create": (C.c_int, [_P, C.POINTER(OdomConfigC), _P, C.POINTER(_P)]),
    "sb_odom_free": (None, [_P]),
    "sb_odom_reserve": (C.c_int, [_P, C.c_int64]),
    "sb_odom_set_pose": (C.c_int, [_P, _D]),
    "sb_odom_get_pose": (C.c_int, [_P, _D]),
    "sb_odom_push": (C.c_int, [_P, _D, C.c_int64, C.c_int32, C.c_int32, C.POINTER(OdomFrameC), _D, C.POINTER(C.c_float),
                               _D, C.POINTER(LoopResultC), C.c_int32]),
    "sb_odom_push_f32": (C.c_int, [_P, _P, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.POINTER(OdomFrameC), _D,
                                   C.POINTER(C.c_float), _D, C.POINTER(LoopResultC), C.c_int32]),
    "sb_map_create": (C.c_int, [_P, _P, C.POINTER(_P)]),
    "sb_map_free": (None, [_P]),
    "sb_map_reserve": (C.c_int, [_P, C.c_int64, C.c_int64, C.c_int64]),
    "sb_map_size": (C.c_int64, [_P]),
    "sb_map_rows": (C.c_int64, [_P]),
    "sb_map_capacity": (C.c_int, [_P, _I64]),
    "sb_map_clear": (C.c_int, [_P]),
    "sb_map_add": (C.c_int, [_P, _D, C.c_int64, _D]),
    "sb_map_set_poses": (C.c_int, [_P, C.c_int32, C.c_int32, _D]),
    "sb_map_get_poses": (C.c_int, [_P, C.c_int32, C.c_int32, _D]),
    "sb_map_occupancy_cells": (C.c_int, [_P, _I32, C.c_int64, _I64]),
    "sb_map_world_f32": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_float), _I64]),
    "sb_map_global": (C.c_int, [_P, C.c_double, _D, _I64]),
    "sb_map_global_f32": (C.c_int, [_P, C.c_double, C.POINTER(C.c_float), _I64]),
    "sb_odom_create2": (C.c_int, [_P, C.POINTER(OdomConfigC), _P, _P, C.POINTER(_P)]),
    "sb_odom_push_many": (C.c_int, [_P, C.c_int32, _P, _I64, _I32, _I32, C.POINTER(OdomFrameC), _P, _P, _P, _P, _I32]),
    "sb_odom_push_many_f32": (C.c_int, [_P, C.c_int32, _P, C.c_int32, _I64, _I32, _I32, C.POINTER(OdomFrameC), _P, _P, _P,
                                        _P, _I32]),
    "sb_gather_results": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(ICPResultC), C.c_int32, C.POINTER(ICPResultC)]),
    "sb_gather_candidates": (C.c_int, [_P, _P, C.c_int32, _D, _I32, C.c_int32, C.c_int32, _D, _I32, _I32]),
    "sb_odometry_factors": (C.c_int, [_P, C.POINTER(ICPResultC), C.c_int32, C.c_int32, C.c_double, C.POINTER(PoseFactorC)]),
    "sb_loop_factors": (C.c_int, [_P, C.POINTER(LoopResultC), C.c_int32, C.POINTER(PoseFactorC)]),
    "sb_default_grid_config": (None, [_P]),
    "sb_transform_clouds": (C.c_int, [_P, _D, _I64, C.c_int32, _D, _D]),
    "sb_occupancy_cells": (C.c_int, [_P, _D, _I64, C.c_int32, _D, _P, _I32, C.c_int64, _I64]),
    "sb_global_map": (C.c_int, [_P, _D, _I64, C.c_int32, _D, C.c_double, _D, _I64]),
    "sb_transform_clouds_f32": (C.c_int, [_P, _D, _I64, C.c_int32, _D, C.POINTER(C.c_float)]),
    "sb_global_map_f32": (C.c_int, [_P, _D, _I64, C.c_int32, _D, C.c_double, C.POINTER(C.c_float), _I64]),
    "sb_synth_scans_dev": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                     C.POINTER(C.c_float), C.c_int32, _D, C.c_int32, C.c_uint64, _P, _I64]),
}

_lib = None


def load_library(path=None):
    """Loads libslam_b200.so and binds every declared symbol.  Raises if the library or a symbol is missing."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or _LIB_PATH
    if not os.path.exists(p):
        raise SlamB200Error(4, f"{p} not found: build it with `make -C lidar-slam-from-scratch_b200` "
                               "(there is no CPU fallback)")
    lib = C.CDLL(p)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def _dp(a):
    return a.ctypes.data_as(_D)


def _f64(a, cols=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if cols is not None:
        a = a.reshape(-1, cols)
    return a


class Engine:
    """One sb_ctx (device, stream, workspace).  Use from one thread at a time."""

    def __init__(self, device=0, stream=None):
        self.lib = load_library()
        h = _P()
        s = self.lib.sb_ctx_create(device, _P(stream) if stream else None, C.byref(h))
        if s != 0:
            raise SlamB200Error(s, "sb_ctx_create failed (needs an sm_100-class GPU; there is no CPU fallback)")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.sb_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, s):
        if s != 0:
            raise SlamB200Error(s, self.lib.sb_last_error(self.h).decode())

    def synchronize(self):
        self._check(self.lib.sb_ctx_synchronize(self.h))

    @property
    def launch_count(self):
        return int(self.lib.sb_ctx_launch_count(self.h))

    STAGES = ("h2d", "voxel", "scan_context", "index_build", "normals", "icp_loop", "d2h")

    def set_profiling(self, on):
        self._check(self.lib.sb_ctx_set_profiling(self.h, 1 if on else 0))

    def stage_ms(self):
        ms = np.zeros(7)
        self._check(self.lib.sb_ctx_stage_ms(self.h, _dp(ms)))
        return dict(zip(self.STAGES, ms.tolist()))

    def stage_host_ms(self):
        ms = np.zeros(7)
        self._check(self.lib.sb_ctx_stage_host_ms(self.h, _dp(ms)))
        return dict(zip(self.STAGES, ms.tolist()))

    def last_counts(self):
        c = np.zeros(5, dtype=np.int64)
        self._check(self.lib.sb_ctx_last_counts(self.h, c.ctypes.data_as(_I64)))
        return dict(raw_rows=int(c[0]), voxel_rows=int(c[1]), target_rows=int(c[2]), nn_queries=int(c[3]),
                    icp_iter_launches=int(c[4]))

    @property
    def last_voxel_path(self):
        """1 = hashed fixed-point sums (float32-born scans), 2 = sort-based; same rows either way."""
        return int(self.lib.sb_ctx_last_voxel_path(self.h))

    # ---- config helpers
    def icp_config(self, max_iterations=50, tolerance=1e-6, min_error=1e-9, initial_transform=None, normals_k=20):
        cfg = ICPConfigC()
        self.lib.sb_default_icp_config(C.byref(cfg))
        cfg.max_iterations = max_iterations
        cfg.tolerance = tolerance
        cfg.min_error = min_error
        cfg.normals_k = normals_k
        if initial_transform is not None:
            T = _f64(initial_transform).reshape(16)
            for i in range(16):
                cfg.initial_transform[i] = T[i]
        return cfg

    # ---- voxel grid (file_utils.cpp:148-196)
    def voxel_downsample(self, points, voxel, return_keys=False):
        pts = _f64(points, 3)
        n = pts.shape[0]
        out = np.empty((max(n, 1), 3))
        keys = np.empty((max(n, 1), 3), dtype=np.int64) if return_keys else None
        m = C.c_int64(0)
        self._check(self.lib.sb_voxel_downsample(self.h, _dp(pts), n, float(voxel), _dp(out), C.byref(m),
                                                 keys.ctypes.data_as(_I64) if return_keys else None))
        if return_keys:
            return out[:m.value].copy(), keys[:m.value].copy()
        return out[:m.value].copy()

    def voxel_downsample_batch_f32(self, points, offsets, voxel, return_keys=False):
        """float32 rows (n x 3 or n x 4) widened on the device; same rows as voxel_downsample_batch of the widened input."""
        pts = np.ascontiguousarray(points, dtype=np.float32)
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        nc = off.shape[0] - 1
        out = np.empty((max(pts.shape[0], 1), 3))
        keys = np.empty((max(pts.shape[0], 1), 3), dtype=np.int64) if return_keys else None
        out_off = np.zeros(nc + 1, dtype=np.int64)
        self._check(self.lib.sb_voxel_downsample_batch_f32(self.h, _P(pts.ctypes.data), int(pts.shape[1]),
                                                           off.ctypes.data_as(_I64), nc, float(voxel), _dp(out),
                                                           out_off.ctypes.data_as(_I64),
                                                           keys.ctypes.data_as(_I64) if return_keys else None))
        m = int(out_off[-1])
        return (out[:m], out_off, keys[:m]) if return_keys else (out[:m], out_off)

    def voxel_downsample_batch(self, points, offsets, voxel, return_keys=False):
        pts = _f64(points, 3)
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        nc = off.shape[0] - 1
        n = int(off[-1])
        out = np.empty((max(n, 1), 3))
        out_off = np.zeros(nc + 1, dtype=np.int64)
        keys = np.empty((max(n, 1), 3), dtype=np.int64) if return_keys else None
        self._check(self.lib.sb_voxel_downsample_batch(self.h, _dp(pts), off.ctypes.data_as(_I64), nc, float(voxel),
                                                       _dp(out), out_off.ctypes.data_as(_I64),
                                                       keys.ctypes.data_as(_I64) if return_keys else None))
        m = int(out_off[-1])
        if return_keys:
            return out[:m].copy(), out_off, keys[:m].copy()
        return out[:m].copy(), out_off

    # ---- ICP (icp.hpp:89-258)
    def solve_point_to_plane(self, source, target, normals):
        s, t, nn = _f64(source, 3), _f64(target, 3), _f64(normals, 3)
        T = np.empty(16)
        self._check(self.lib.sb_solve_point_to_plane(self.h, _dp(s), _dp(t), _dp(nn), s.shape[0], _dp(T)))
        return T.reshape(4, 4)

    def icp_point_to_plane(self, source, target, cfg=None):
        s, t = _f64(source, 3), _f64(target, 3)
        cfg = cfg or self.icp_config()
        res = ICPResultC()
        self._check(self.lib.sb_icp_point_to_plane(self.h, _dp(s), s.shape[0], _dp(t), t.shape[0], C.byref(cfg),
                                                   C.byref(res)))
        return ICPResult(res)

    def register_batch(self, points, offsets, pair_src, pair_tgt, voxel=0.0, cfg=None, want_sc=False, device_ptr=None):
        """Batched pair registration (sb_register_batch / _dev).  device_ptr: raw device pointer to the xyz rows."""
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        nc = off.shape[0] - 1
        ps = np.ascontiguousarray(pair_src, dtype=np.int32)
        pt = np.ascontiguousarray(pair_tgt, dtype=np.int32)
        npairs = ps.shape[0]
        cfg = cfg or self.icp_config()
        res = np.zeros(max(npairs, 1), dtype=ICP_DTYPE)
        rp = res.ctypes.data_as(C.POINTER(ICPResultC))
        sc = np.empty((nc, SB_SC_SIZE)) if want_sc else None
        if device_ptr is None and isinstance(points, np.ndarray) and points.dtype == np.float32:
            # float32 records as they are on disk (rows of 3 or 4 floats: xyz / KITTI xyzi), widened on the device
            pts = np.ascontiguousarray(points)
            s = self.lib.sb_register_batch_f32(self.h, _P(pts.ctypes.data), int(pts.shape[1]), off.ctypes.data_as(_I64),
                                               nc, float(voxel), ps.ctypes.data_as(_I32), pt.ctypes.data_as(_I32),
                                               npairs, C.byref(cfg), rp, _dp(sc) if want_sc else None)
        elif device_ptr is None:
            pts = _f64(points, 3)
            s = self.lib.sb_register_batch(self.h, _dp(pts), off.ctypes.data_as(_I64), nc, float(voxel),
                                           ps.ctypes.data_as(_I32), pt.ctypes.data_as(_I32), npairs, C.byref(cfg), rp,
                                           _dp(sc) if want_sc else None)
        else:
            s = self.lib.sb_register_batch_dev(self.h, _P(device_ptr), off.ctypes.data_as(_I64), nc, float(voxel),
                                               ps.ctypes.data_as(_I32), pt.ctypes.data_as(_I32), npairs, C.byref(cfg),
                                               rp, _dp(sc) if want_sc else None)
        self._check(s)
        out = ICPResultBatch(res[:npairs])
        return (out, sc) if want_sc else out

    # ---- after the path: world-frame clouds, occupancy cells, global map (slam_node.cpp:147-152, 196-238)
    def odometry_poses(self, results, max_error=1.0, initial_pose=None):
        """slam_node.cpp:139-145: absolute poses (n + 1, 4, 4) of a sequence from its frame-to-frame registrations."""
        rec = np.ascontiguousarray(results.rec)
        n = rec.shape[0]
        out = np.empty((n + 1, 16))
        p0 = None if initial_pose is None else np.ascontiguousarray(initial_pose, dtype=np.float64).reshape(16)
        self._check(self.lib.sb_odometry_poses(self.h, rec.ctypes.data_as(C.POINTER(ICPResultC)), n, float(max_error),
                                               _dp(p0) if p0 is not None else None, _dp(out)))
        return out.reshape(n + 1, 4, 4)

    def odometry_factors(self, results, first_frame=0, max_error=1.0):
        """slam_node.cpp:139-145 for a batch: the (from, to, relative, fitness, noise scale) records the node hands to
        PoseGraph::addOdometryFactor (pose_graph.cpp:81-117), as a structured array (FACTOR_DTYPE)."""
        rec = np.ascontiguousarray(results.rec)
        out = np.zeros(rec.shape[0], dtype=FACTOR_DTYPE)
        self._check(self.lib.sb_odometry_factors(self.h, rec.ctypes.data_as(C.POINTER(ICPResultC)), rec.shape[0],
                                                 int(first_frame), float(max_error),
                                                 out.ctypes.data_as(C.POINTER(PoseFactorC))))
        return out

    def loop_factors(self, loop_results):
        """slam_node.cpp:163-167: accepted loop closures (list of dicts as LoopClosureDetector.detect returns them, or a
        ctypes array of LoopResultC) -> addLoopClosure(match, query, transform) records."""
        if isinstance(loop_results, (list, tuple)):
            arr = (LoopResultC * max(len(loop_results), 1))()
            for i, r in enumerate(loop_results):
                arr[i].query_frame, arr[i].match_frame = int(r["query_frame"]), int(r["match_frame"])
                arr[i].transform[:] = list(np.asarray(r["transform"], dtype=np.float64).reshape(16))
                arr[i].scan_context_distance = float(r["scan_context_distance"])
                arr[i].icp_fitness = float(r["icp_fitness"])
            n = len(loop_results)
        else:
            arr, n = loop_results, len(loop_results)
        out = np.zeros(n, dtype=FACTOR_DTYPE)
        self._check(self.lib.sb_loop_factors(self.h, arr, n, out.ctypes.data_as(C.POINTER(PoseFactorC))))
        return out

    def transform_clouds(self, points, offsets, poses):
        pts, off = _f64(points, 3), np.ascontiguousarray(offsets, dtype=np.int64)
        T = np.ascontiguousarray(poses, dtype=np.float64).reshape(-1, 16)
        out = np.empty_like(pts)
        self._check(self.lib.sb_transform_clouds(self.h, _dp(pts), off.ctypes.data_as(_I64), off.shape[0] - 1, _dp(T),
                                                 _dp(out)))
        return out

    def occupancy_cells(self, points, offsets, poses, resolution=0.2, height_min=0.3, height_max=2.0, max_range=40.0,
                        capacity=None):
        pts, off = _f64(points, 3), np.ascontiguousarray(offsets, dtype=np.int64)
        T = np.ascontiguousarray(poses, dtype=np.float64).reshape(-1, 16)
        cfg = (C.c_double * 4)(resolution, height_min, height_max, max_range)
        cap = int(capacity if capacity is not None else max(pts.shape[0], 1))
        cells = np.empty((max(cap, 1), 2), dtype=np.int32)
        cnt = C.c_int64(0)
        self._check(self.lib.sb_occupancy_cells(self.h, _dp(pts), off.ctypes.data_as(_I64), off.shape[0] - 1, _dp(T),
                                                C.cast(cfg, _P), cells.ctypes.data_as(_I32), cap, C.byref(cnt)))
        return cells[:min(cnt.value, cap)].copy(), int(cnt.value)

    def global_map(self, points, offsets, poses, voxel):
        pts, off = _f64(points, 3), np.ascontiguousarray(offsets, dtype=np.int64)
        T = np.ascontiguousarray(poses, dtype=np.float64).reshape(-1, 16)
        out = np.empty((max(pts.shape[0], 1), 3))
        m = C.c_int64(0)
        self._check(self.lib.sb_global_map(self.h, _dp(pts), off.ctypes.data_as(_I64), off.shape[0] - 1, _dp(T),
                                           float(voxel), _dp(out), C.byref(m)))
        return out[:m.value].copy()

    def transform_clouds_f32(self, points, offsets, poses):
        """World-frame clouds as PointCloud2 float32 xyz records (slam_node.cpp:147, 299-322)."""
        pts, off = _f64(points, 3), np.ascontiguousarray(offsets, dtype=np.int64)
        T = np.ascontiguousarray(poses, dtype=np.float64).reshape(-1, 16)
        out = np.empty(pts.shape, dtype=np.float32)
        self._check(self.lib.sb_transform_clouds_f32(self.h, _dp(pts), off.ctypes.data_as(_I64), off.shape[0] - 1,
                                                     _dp(T), out.ctypes.data_as(C.POINTER(C.c_float))))
        return out

    def global_map_f32(self, points, offsets, poses, voxel):
        """Global map as PointCloud2 float32 xyz records (slam_node.cpp:235-238, 299-322)."""
        pts, off = _f64(points, 3), np.ascontiguousarray(offsets, dtype=np.int64)
        T = np.ascontiguousarray(poses, dtype=np.float64).reshape(-1, 16)
        out = np.empty((max(pts.shape[0], 1), 3), dtype=np.float32)
        m = C.c_int64(0)
        self._check(self.lib.sb_global_map_f32(self.h, _dp(pts), off.ctypes.data_as(_I64), off.shape[0] - 1, _dp(T),
                                               float(voxel), out.ctypes.data_as(C.POINTER(C.c_float)), C.byref(m)))
        return out[:m.value].copy()

    # ---- Scan Context (scan_context.hpp)
    def sc_compute(self, cloud):
        pts = _f64(cloud, 3)
        d = np.empty(SB_SC_SIZE)
        self._check(self.lib.sb_sc_compute(self.h, _dp(pts), pts.shape[0], _dp(d)))
        return d

    def sc_distance(self, a, b):
        a, b = _f64(a).reshape(-1), _f64(b).reshape(-1)
        out = C.c_double(0)
        self._check(self.lib.sb_sc_distance(self.h, _dp(a), _dp(b), C.byref(out)))
        return out.value

    def sc_distance_batch(self, query, db):
        q, d = _f64(query).reshape(-1), _f64(db).reshape(-1, SB_SC_SIZE)
        out = np.empty(max(d.shape[0], 1))
        self._check(self.lib.sb_sc_distance_batch(self.h, _dp(q), _dp(d), d.shape[0], _dp(out)))
        return out[:d.shape[0]]

    def sc_keys(self, desc):
        d = _f64(desc).reshape(-1)
        r, s = np.empty(20), np.empty(60)
        self._check(self.lib.sb_sc_keys(self.h, _dp(d), _dp(r), _dp(s)))
        return r, s

    # ---- synthetic scans straight into device memory (bench input generator)
    def synth_scans_dev(self, sensor, boxes, poses, noise_seed, d_xyz_ptr):
        b = np.ascontiguousarray(boxes, dtype=np.float32).reshape(-1, 6)
        p = _f64(poses, 3)
        off = np.zeros(p.shape[0] + 1, dtype=np.int64)
        self._check(self.lib.sb_synth_scans_dev(self.h, sensor["beams"], sensor["azimuth_steps"], sensor["elev_top_deg"],
                                                sensor["elev_bot_deg"], sensor["max_range"], sensor["noise_sigma"],
                                                sensor["sensor_height"], b.ctypes.data_as(C.POINTER(C.c_float)),
                                                b.shape[0], _dp(p), p.shape[0], int(noise_seed), _P(d_xyz_ptr),
                                                off.ctypes.data_as(_I64)))
        return off


ICP_DTYPE = np.dtype([("transformation", "f8", (16,)), ("final_error", "f8"), ("converged", "i4"),
                      ("num_iterations", "i4"), ("history_len", "i4"), ("status", "i4"),
                      ("error_history", "f8", (SB_MAX_ICP_ITERATIONS + 1,))])
assert ICP_DTYPE.itemsize == C.sizeof(ICPResultC)


class ICPResult:
    """slam::ICPResult (types.hpp:155-164)."""

    def __init__(self, r):
        if isinstance(r, np.void):  # one record of an ICP_DTYPE array
            self.transformation = r["transformation"].reshape(4, 4).copy()
            self.converged = bool(r["converged"])
            self.num_iterations = int(r["num_iterations"])
            self.final_error = float(r["final_error"])
            self.error_history = r["error_history"][:int(r["history_len"])].copy()
            self.status = int(r["status"])
            return
        self.transformation = np.array(r.transformation[:]).reshape(4, 4)
        self.converged = bool(r.converged)
        self.num_iterations = int(r.num_iterations)
        self.final_error = float(r.final_error)
        self.error_history = np.array(r.error_history[:r.history_len])
        self.status = int(r.status)

    def success(self):  # types.hpp:162
        return self.converged and self.final_error < 0.1


class ICPResultBatch:
    """The sb_icp_result records of one sb_register_batch call, kept as one structured array (no per-pair Python
    objects on the hot path); indexing yields an ICPResult."""

    def __init__(self, rec):
        self.rec = rec

    def __len__(self):
        return self.rec.shape[0]

    def __getitem__(self, i):
        return ICPResult(self.rec[i])

    def __iter__(self):
        return (ICPResult(self.rec[i]) for i in range(len(self)))

    @property
    def transformations(self):
        return self.rec["transformation"].reshape(-1, 4, 4)

    @property
    def num_iterations(self):
        return self.rec["num_iterations"]

    @property
    def converged(self):
        return self.rec["converged"].astype(bool)

    @property
    def final_errors(self):
        return self.rec["final_error"]

    @property
    def status(self):
        return self.rec["status"]

    def records20(self):
        """(n, 20) float64: T[16], final_error, num_iterations, converged, status — the NCCL gather payload."""
        out = np.empty((len(self), 20))
        out[:, :16] = self.rec["transformation"]
        out[:, 16] = self.rec["final_error"]
        out[:, 17] = self.rec["num_iterations"]
        out[:, 18] = self.rec["converged"]
        out[:, 19] = self.rec["status"]
        return out


class KDTree:
    """slam::KDTree (kdtree.hpp:18-186) — backed by the GPU box-tree index."""

    def __init__(self, engine, points):
        self.e = engine
        pts = _f64(points, 3)
        self.n = pts.shape[0]
        h = _P()
        engine._check(engine.lib.sb_index_build(engine.h, _dp(pts), self.n, C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            if self.e.h:   # after Engine.close() its context is gone: freeing would touch it, so the handle is dropped
                self.e.lib.sb_index_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def size(self):
        return int(self.e.lib.sb_index_size(self.h))

    def nearest_batch(self, queries):
        q = _f64(queries, 3)
        idx = np.empty(max(q.shape[0], 1), dtype=np.int32)
        d2 = np.empty(max(q.shape[0], 1))
        self.e._check(self.e.lib.sb_index_nearest_batch(self.h, _dp(q), q.shape[0], idx.ctypes.data_as(_I32), _dp(d2)))
        return idx[:q.shape[0]], d2[:q.shape[0]]

    def nearest(self, query):
        i, d = self.nearest_batch(np.asarray(query).reshape(1, 3))
        return int(i[0]), float(d[0])

    def k_nearest_batch(self, queries, k):
        q = _f64(queries, 3)
        idx = np.empty((max(q.shape[0], 1), k), dtype=np.int32)
        d2 = np.empty((max(q.shape[0], 1), k))
        self.e._check(self.e.lib.sb_index_knn(self.h, _dp(q), q.shape[0], k, idx.ctypes.data_as(_I32), _dp(d2)))
        return idx[:q.shape[0]], d2[:q.shape[0]]

    def k_nearest(self, query, k):
        i, _ = self.k_nearest_batch(np.asarray(query).reshape(1, 3), k)
        return [int(v) for v in i[0] if v >= 0]

    def find_correspondences(self, source):  # NearestNeighborSearch::find_correspondences, kdtree.hpp:198-214
        s = _f64(source, 3)
        m = np.empty((max(s.shape[0], 1), 3))
        d = np.empty(max(s.shape[0], 1))
        self.e._check(self.e.lib.sb_index_find_correspondences(self.h, _dp(s), s.shape[0], _dp(m), _dp(d)))
        return m[:s.shape[0]], d[:s.shape[0]]

    def estimate_normals(self, k=20, return_evals=False):
        n = self.size()
        out = np.empty((max(n, 1), 3))
        ev = np.empty((max(n, 1), 3)) if return_evals else None
        self.e._check(self.e.lib.sb_estimate_normals(self.h, k, _dp(out), _dp(ev) if return_evals else None))
        return (out[:n], ev[:n]) if return_evals else out[:n]


def estimate_normals(points, tree, k=20):
    """slam::estimate_normals(points, tree, k) (icp.hpp:23-67); `points` must be the cloud the tree indexes."""
    return tree.estimate_normals(k)


class LoopClosureDetector:
    """slam::LoopClosureDetector (loop_closure.hpp:41-149)."""

    def __init__(self, engine, frame_gap=50, sc_distance_threshold=0.25, icp_fitness_threshold=0.3, max_candidates=3,
                 rank=0, world=1, verify_chunk=0, icp_max_iterations=30, normals_k=20):
        self.e = engine
        cfg = LoopConfigC()
        engine.lib.sb_default_loop_config(C.byref(cfg))
        cfg.frame_gap = frame_gap
        cfg.sc_distance_threshold = sc_distance_threshold
        cfg.icp_fitness_threshold = icp_fitness_threshold
        cfg.max_candidates = max_candidates
        cfg.verify_chunk = verify_chunk
        cfg.icp_max_iterations = icp_max_iterations
        cfg.normals_k = normals_k
        self.cfg = cfg
        h = _P()
        engine._check(engine.lib.sb_loop_create(engine.h, C.byref(cfg), rank, world, C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            if self.e.h:   # after Engine.close() its context is gone: freeing would touch it, so the handle is dropped
                self.e.lib.sb_loop_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def addFrame(self, points, frame_idx, desc=None):
        p = _f64(points, 3)
        if desc is None:
            self.e._check(self.e.lib.sb_loop_add_frame(self.h, _dp(p), p.shape[0], frame_idx))
        else:
            d = _f64(desc).reshape(-1)
            self.e._check(self.e.lib.sb_loop_add_frame_desc(self.h, _dp(p), p.shape[0], frame_idx, _dp(d)))

    def reserve(self, n_entries, total_rows):
        """Size the device pools up front (no counterpart in the reference: its std::vectors grow on the host)."""
        self.e._check(self.e.lib.sb_loop_reserve(self.h, int(n_entries), int(total_rows)))

    def size(self):
        return int(self.e.lib.sb_loop_size(self.h))

    def clear(self):
        self.e._check(self.e.lib.sb_loop_clear(self.h))

    @staticmethod
    def _result(r):
        return dict(query_frame=r.query_frame, match_frame=r.match_frame,
                    transform=np.array(r.transform[:]).reshape(4, 4), scan_context_distance=r.scan_context_distance,
                    icp_fitness=r.icp_fitness)

    def detect(self, capacity=64):
        res = (LoopResultC * capacity)()
        cnt = C.c_int32(0)
        self.e._check(self.e.lib.sb_loop_detect(self.h, res, capacity, C.byref(cnt)))
        return [self._result(res[i]) for i in range(min(cnt.value, capacity))]

    def candidates_local(self, capacity=4096):
        dist = np.empty(max(capacity, 1))
        ent = np.empty(max(capacity, 1), dtype=np.int32)
        cnt = C.c_int32(0)
        self.e._check(self.e.lib.sb_loop_candidates_local(self.h, _dp(dist), ent.ctypes.data_as(_I32), capacity,
                                                          C.byref(cnt)))
        m = min(cnt.value, capacity)
        return dist[:m].copy(), ent[:m].copy()

    def verify_entries(self, entries, dist):
        ent = np.ascontiguousarray(entries, dtype=np.int32)
        d = _f64(dist).reshape(-1)
        n = ent.shape[0]
        res = (LoopResultC * max(n, 1))()
        conv = np.zeros(max(n, 1), dtype=np.int32)
        self.e._check(self.e.lib.sb_loop_verify_entries(self.h, ent.ctypes.data_as(_I32), _dp(d), n, res,
                                                        conv.ctypes.data_as(_I32)))
        return [self._result(res[i]) for i in range(n)], conv[:n].astype(bool)

    def addFrames(self, xyz, offsets, frame_idx, descs=None):
        """addFrame for every cloud of a CSR batch (cloud f = rows offsets[f]:offsets[f+1]) in one call; descs: optional
        (n_frames, 1200) Scan Context descriptors.  Same detector state as one addFrame per cloud."""
        p = _f64(xyz, 3)
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        fi = np.ascontiguousarray(frame_idx, dtype=np.int32)
        n = off.shape[0] - 1
        if fi.shape[0] != n:
            raise ValueError("frame_idx needs one frame per cloud")
        d = None if descs is None else _f64(descs).reshape(n, SB_SC_SIZE)
        self.e._check(self.e.lib.sb_loop_add_frames(self.h, _dp(p), off.ctypes.data_as(_I64), n, fi.ctypes.data_as(_I32),
                                                    _dp(d) if d is not None else None))

    def candidates_batch(self, query_entries, k=SB_LOOP_SELECT_MAX):
        """Stage 1 of detect() for every listed query entry (strictly ascending): per query the best min(k, count)
        (distance, entry) pairs as arrays, and the number of candidates under the threshold."""
        q = np.ascontiguousarray(query_entries, dtype=np.int32)
        n = q.shape[0]
        dist = np.empty((max(n, 1), k))
        ent = np.empty((max(n, 1), k), dtype=np.int32)
        cnt = np.zeros(max(n, 1), dtype=np.int32)
        self.e._check(self.e.lib.sb_loop_candidates_batch(self.h, q.ctypes.data_as(_I32), n, int(k), _dp(dist),
                                                          ent.ctypes.data_as(_I32), cnt.ctypes.data_as(_I32)))
        return [(dist[i, :min(cnt[i], k)].copy(), ent[i, :min(cnt[i], k)].copy()) for i in range(n)], cnt[:n].copy()

    def detect_batch(self, query_entries):
        """detect() as it would have answered right after each listed entry (strictly ascending) was added: a list of
        per-query lists of the dicts detect() returns."""
        q = np.ascontiguousarray(query_entries, dtype=np.int32)
        n = q.shape[0]
        m = max(int(self.cfg.max_candidates), 0)
        res = (LoopResultC * max(n * m, 1))()
        cnt = np.zeros(max(n, 1), dtype=np.int32)
        self.e._check(self.e.lib.sb_loop_detect_batch(self.h, q.ctypes.data_as(_I32), n, res, cnt.ctypes.data_as(_I32)))
        return [[self._result(res[i * m + j]) for j in range(cnt[i])] for i in range(n)]


def _across_args(dbs, queries):
    if len(dbs) == 0:
        raise ValueError("no detectors")
    q = np.asarray(queries, dtype=np.int32).reshape(-1, 2) if len(queries) else np.zeros((0, 2), dtype=np.int32)
    qdb = np.ascontiguousarray(q[:, 0])
    qe = np.ascontiguousarray(q[:, 1])
    hs = (_P * len(dbs))(*[d.h for d in dbs])
    return dbs[0].e, hs, qdb, qe, q.shape[0]


def candidates_across(dbs, queries, k=SB_LOOP_SELECT_MAX):
    """Stage 1 of detect() across detectors (sb_loop_candidates_across).  dbs: LoopClosureDetector objects of one engine
    (world 1, one loop config); queries: (db_index, entry) pairs.  Query i is searched against every entry of every
    other detector, without a frame gap.  Returns per query the best min(k, count) candidates as arrays (dist, db,
    entry), ascending by (distance, db, entry), and the number of candidates under the threshold."""
    e, hs, qdb, qe, n = _across_args(dbs, queries)
    dist = np.empty((max(n, 1), k))
    db = np.empty((max(n, 1), k), dtype=np.int32)
    ent = np.empty((max(n, 1), k), dtype=np.int32)
    cnt = np.zeros(max(n, 1), dtype=np.int32)
    e._check(e.lib.sb_loop_candidates_across(hs, len(dbs), qdb.ctypes.data_as(_I32), qe.ctypes.data_as(_I32), n, int(k),
                                             _dp(dist), db.ctypes.data_as(_I32), ent.ctypes.data_as(_I32),
                                             cnt.ctypes.data_as(_I32)))
    out = []
    for i in range(n):
        m = min(int(cnt[i]), k)
        out.append((dist[i, :m].copy(), db[i, :m].copy(), ent[i, :m].copy()))
    return out, cnt[:n].copy()


def detect_across(dbs, queries):
    """detect() across detectors (sb_loop_detect_across): per query the list of accepted loops, dicts as
    LoopClosureDetector.detect returns them plus match_db, the index in dbs of the matched entry's detector
    (match_frame is that entry's frame, query_frame the query entry's)."""
    e, hs, qdb, qe, n = _across_args(dbs, queries)
    m = max(int(dbs[0].cfg.max_candidates), 0)
    res = (LoopResultC * max(n * m, 1))()
    mdb = np.zeros(max(n * m, 1), dtype=np.int32)
    cnt = np.zeros(max(n, 1), dtype=np.int32)
    e._check(e.lib.sb_loop_detect_across(hs, len(dbs), qdb.ctypes.data_as(_I32), qe.ctypes.data_as(_I32), n, res,
                                         mdb.ctypes.data_as(_I32), cnt.ctypes.data_as(_I32)))
    return [[dict(LoopClosureDetector._result(res[i * m + j]), match_db=int(mdb[i * m + j])) for j in range(cnt[i])]
            for i in range(n)]


class OdomFrame:
    """What Odometry.push returns for one frame: frame_idx, state (ODOM_FIRST / ODOM_REGISTERED / ODOM_SKIPPED),
    n_points, pose (4x4), icp (ICPResult, registered frames only), loops (accepted loop closures, dicts as
    LoopClosureDetector.detect returns them) and the outputs asked for: cloud (downsampled rows), world_f32
    (PointCloud2 float32 xyz of the world-frame cloud), desc (Scan Context, 1200)."""

    def __init__(self, f, loops, cloud, world_f32, desc):
        self.frame_idx = int(f.frame_idx)
        self.state = int(f.state)
        self.n_points = int(f.n_points)
        self.pose = np.array(f.pose[:]).reshape(4, 4)
        self.icp = ICPResult(f.icp) if self.state == ODOM_REGISTERED else None
        self.n_loops = int(f.n_loops)
        self.loops = loops
        self.cloud, self.world_f32, self.desc = cloud, world_f32, desc


class Odometry:
    """Streaming odometry session (sb_odom_*): SlamNode::process_frame (slam_node.cpp:118-175) one scan per call, with
    the previous frame's cloud, index and normals kept on the device.  loop: an optional LoopClosureDetector, map: an
    optional Map, both on the same engine and open while the session is."""

    def __init__(self, engine, voxel=0.5, cfg=None, max_error=1.0, min_points=1000, initial_pose=None, loop=None,
                 map=None):
        self.e = engine
        self.loop = loop
        self.map = map
        c = OdomConfigC()
        engine.lib.sb_default_odom_config(C.byref(c))
        c.voxel = float(voxel)
        c.min_points = int(min_points)
        c.max_error = float(max_error)
        if cfg is not None:
            c.icp = cfg
        if initial_pose is not None:
            c.initial_pose[:] = list(_f64(initial_pose).reshape(16))
        self.cfg = c
        h = _P()
        engine._check(engine.lib.sb_odom_create2(engine.h, C.byref(c), loop.h if loop is not None else None,
                                                 map.h if map is not None else None, C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            if self.e.h:   # after Engine.close() its context is gone: freeing would touch it, so the handle is dropped
                self.e.lib.sb_odom_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reserve(self, max_raw_rows):
        """Size every buffer for frames of up to max_raw_rows rows, so that no later push allocates."""
        self.e._check(self.e.lib.sb_odom_reserve(self.h, int(max_raw_rows)))

    def set_pose(self, pose):
        """Continue the pose chain from `pose` (4x4), e.g. after a pose-graph optimisation (slam_node.cpp:177-185)."""
        p = _f64(pose).reshape(16)
        self.e._check(self.e.lib.sb_odom_set_pose(self.h, _dp(p)))

    @property
    def pose(self):
        p = np.empty(16)
        self.e._check(self.e.lib.sb_odom_get_pose(self.h, _dp(p)))
        return p.reshape(4, 4)

    def push(self, points, frame_idx, add_frame=True, detect=False, want_cloud=False, want_world_f32=False,
             want_desc=False, add_map=True):
        """One frame.  points: (n, 3) float64 rows, or float32 records (n, 3) / (n, 4) as read from PLY / KITTI files
        (widened on the device).  add_frame adds the frame to the attached detector (ignored without one); detect runs
        its detect() (needs a detector); add_map adds the frame to the attached map (ignored without one: a skipped
        frame as an entry with no rows and the repeated pose).  Returns an OdomFrame."""
        f32 = isinstance(points, np.ndarray) and points.dtype == np.float32
        if f32:
            pts = np.ascontiguousarray(points)
            if pts.ndim != 2:
                raise ValueError("float32 points must be (n, 3) or (n, 4) records")
        else:
            pts = _f64(points, 3)
        n = pts.shape[0]
        flags = ((ODOM_ADD_FRAME if add_frame and self.loop is not None else 0) | (ODOM_DETECT if detect else 0) |
                 (ODOM_ADD_MAP if add_map and self.map is not None else 0))
        cloud = np.empty((max(n, 1), 3)) if want_cloud else None
        world = np.empty((max(n, 1), 3), dtype=np.float32) if want_world_f32 else None
        desc = np.empty(SB_SC_SIZE) if want_desc else None
        cap = max(int(self.loop.cfg.max_candidates), 0) if (detect and self.loop is not None) else 0
        loops = (LoopResultC * max(cap, 1))()
        fr = OdomFrameC()
        fp = C.POINTER(C.c_float)
        args = (int(frame_idx), flags, C.byref(fr), _dp(cloud) if want_cloud else None,
                world.ctypes.data_as(fp) if want_world_f32 else None, _dp(desc) if want_desc else None, loops, cap)
        if f32:
            s = self.e.lib.sb_odom_push_f32(self.h, _P(pts.ctypes.data), int(pts.shape[1]), n, *args)
        else:
            s = self.e.lib.sb_odom_push(self.h, _dp(pts), n, *args)
        self.e._check(s)
        m = int(fr.n_points)
        state = int(fr.state)
        out_cloud = cloud[:m].copy() if want_cloud else None
        out_world = world[:m].copy() if (want_world_f32 and state != ODOM_SKIPPED) else None
        out_desc = desc if (want_desc and state != ODOM_SKIPPED) else None
        res = [LoopClosureDetector._result(loops[i]) for i in range(min(int(fr.n_loops), cap))]
        return OdomFrame(fr, res, out_cloud, out_world, out_desc)


def push_many(sessions, frames, frame_idx, add_frame=True, detect=False, add_map=True, want_cloud=False,
              want_world_f32=False, want_desc=False, loop_capacity=None):
    """One frame into each of many Odometry sessions of one engine in one call (sb_odom_push_many): one voxel grid, one
    index build and one ICP batch for all of them.  The results are those of sessions[i].push(frames[i], frame_idx[i],
    ...) for i in order, bit for bit, and the sessions are left as those pushes would leave them.  frames: (n, 3)
    float64 rows each, or float32 records of one width for all (n, 3) / (n, 4).  frame_idx, add_frame, detect, add_map
    and loop_capacity (accepted loops returned per session; default: its detector's max_candidates) may be scalars or one
    value per session.  Rules (SlamB200Error SB_ERR_INVALID_ARG otherwise): no session twice, no shared detector or map,
    one voxel and icp config for all.  A call that fails changes no session.  Returns a list of OdomFrame."""
    n = len(sessions)
    if len(frames) != n:
        raise ValueError("one frame per session")
    if n == 0:
        return []
    e = sessions[0].e

    def per(v, name):
        v = list(v) if isinstance(v, (list, tuple, np.ndarray)) else [v] * n
        if len(v) != n:
            raise ValueError(f"{name}: one value per session")
        return v

    idx, af, dt, am = per(frame_idx, "frame_idx"), per(add_frame, "add_frame"), per(detect, "detect"), per(add_map, "add_map")
    f32 = isinstance(frames[0], np.ndarray) and frames[0].dtype == np.float32
    if f32:
        pts = [np.ascontiguousarray(p) for p in frames]
        if any(p.dtype != np.float32 or p.ndim != 2 or p.shape[1] != pts[0].shape[1] for p in pts):
            raise ValueError("float32 frames must all be (n, 3) or all (n, 4) records")
    else:
        pts = [_f64(p, 3) for p in frames]
    rows = np.array([p.shape[0] for p in pts], dtype=np.int64)
    flags = np.array([(ODOM_ADD_FRAME if af[i] and s.loop is not None else 0) | (ODOM_DETECT if dt[i] else 0) |
                      (ODOM_ADD_MAP if am[i] and s.map is not None else 0) for i, s in enumerate(sessions)], dtype=np.int32)
    fi = np.array([int(x) for x in idx], dtype=np.int32)
    caps = per(loop_capacity, "loop_capacity") if loop_capacity is not None else [
        max(int(s.loop.cfg.max_candidates), 0) if (dt[i] and s.loop is not None) else 0 for i, s in enumerate(sessions)]
    cap = np.array([int(c) for c in caps], dtype=np.int32)
    loops = [(LoopResultC * max(int(c), 1))() for c in cap]
    clouds = [np.empty((max(int(r), 1), 3)) for r in rows] if want_cloud else None
    worlds = [np.empty((max(int(r), 1), 3), dtype=np.float32) for r in rows] if want_world_f32 else None
    descs = [np.empty(SB_SC_SIZE) for _ in range(n)] if want_desc else None

    def ptrs(arrs):
        return (_P * n)(*[a.ctypes.data for a in arrs]) if arrs is not None else None

    hs = (_P * n)(*[s.h for s in sessions])
    out = (OdomFrameC * n)()
    tail = (fi.ctypes.data_as(_I32), flags.ctypes.data_as(_I32), out, ptrs(clouds), ptrs(worlds), ptrs(descs),
            (_P * n)(*[C.addressof(l) for l in loops]), cap.ctypes.data_as(_I32))
    xs = ptrs(pts)
    if f32:
        st = e.lib.sb_odom_push_many_f32(hs, n, xs, int(pts[0].shape[1]), rows.ctypes.data_as(_I64), *tail)
    else:
        st = e.lib.sb_odom_push_many(hs, n, xs, rows.ctypes.data_as(_I64), *tail)
    e._check(st)
    res = []
    for i in range(n):
        f = out[i]
        m, state = int(f.n_points), int(f.state)
        lp = [LoopClosureDetector._result(loops[i][j]) for j in range(min(int(f.n_loops), int(cap[i])))]
        res.append(OdomFrame(f, lp, clouds[i][:m].copy() if want_cloud else None,
                             worlds[i][:m].copy() if (want_world_f32 and state != ODOM_SKIPPED) else None,
                             descs[i] if (want_desc and state != ODOM_SKIPPED) else None))
    return res


class Map:
    """Device-resident map (sb_map_*): the node's keyframe clouds (sensor frame), their poses and the occupancy cell set
    (slam_node.cpp:147-157, 177-238).  After a pose-graph optimisation only the poses are uploaded (set_poses); the
    cells, the global map and the world-frame window are rebuilt from the resident clouds, with the bits of
    Engine.occupancy_cells / global_map / transform_clouds_f32 over the same clouds and poses."""

    def __init__(self, engine, resolution=0.2, height_min=0.3, height_max=2.0, max_range=40.0):
        self.e = engine
        self.grid = (C.c_double * 4)(resolution, height_min, height_max, max_range)
        h = _P()
        engine._check(engine.lib.sb_map_create(engine.h, C.cast(self.grid, _P), C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            if self.e.h:   # after Engine.close() its context is gone: freeing would touch it, so the handle is dropped
                self.e.lib.sb_map_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reserve(self, n_entries, total_rows, n_cells):
        """Room for n_entries entries, total_rows rows and n_cells cells: no later call allocates within them."""
        self.e._check(self.e.lib.sb_map_reserve(self.h, int(n_entries), int(total_rows), int(n_cells)))

    def size(self):
        return int(self.e.lib.sb_map_size(self.h))

    def __len__(self):
        return self.size()

    @property
    def rows(self):
        return int(self.e.lib.sb_map_rows(self.h))

    def capacity(self):
        """(entries, rows, cell-table slots) the device buffers hold now."""
        c = np.zeros(3, dtype=np.int64)
        self.e._check(self.e.lib.sb_map_capacity(self.h, c.ctypes.data_as(_I64)))
        return tuple(int(v) for v in c)

    def clear(self):
        self.e._check(self.e.lib.sb_map_clear(self.h))

    def add(self, points, pose):
        """One entry: a sensor-frame cloud (n, 3) and its 4x4 pose; its occupancy cells are inserted at once."""
        p = _f64(points, 3)
        T = _f64(pose)
        if T.size != 16:
            raise ValueError("pose must be a 4x4 matrix")
        self.e._check(self.e.lib.sb_map_add(self.h, _dp(p), p.shape[0], _dp(T.reshape(16))))

    def _range(self, first, n):
        first, n = int(first), int(n)
        if first < 0 or n < 0 or first + n > self.size():
            raise ValueError(f"entries [{first}, {first + n}) outside [0, {self.size()})")
        return first, n

    def set_poses(self, poses, first=0):
        """Replace the poses of entries [first, first + len(poses)) ((k, 4, 4)); the cell set is rebuilt on the device."""
        T = _f64(poses)
        if T.size % 16:
            raise ValueError("poses must be (k, 4, 4)")
        T = T.reshape(-1, 16)
        first, n = self._range(first, T.shape[0])
        self.e._check(self.e.lib.sb_map_set_poses(self.h, first, n, _dp(T)))

    def poses(self, first=0, n=None):
        first, n = self._range(first, self.size() - int(first) if n is None else n)
        out = np.empty((max(n, 1), 16))
        self.e._check(self.e.lib.sb_map_get_poses(self.h, first, n, _dp(out)))
        return out[:n].reshape(n, 4, 4)

    def occupancy_cells(self, capacity=None):
        """(cells (m, 2) int32 ascending in (x, y), count): the first `capacity` cells (all by default) and how many
        there are."""
        if capacity is None:
            cnt = C.c_int64(0)
            self.e._check(self.e.lib.sb_map_occupancy_cells(self.h, None, 0, C.byref(cnt)))
            capacity = cnt.value
        cap = int(capacity)
        if cap < 0:
            raise ValueError("capacity must be >= 0")
        cells = np.empty((max(cap, 1), 2), dtype=np.int32)
        cnt = C.c_int64(0)
        self.e._check(self.e.lib.sb_map_occupancy_cells(self.h, cells.ctypes.data_as(_I32), cap, C.byref(cnt)))
        return cells[:min(cnt.value, cap)].copy(), int(cnt.value)

    def world_f32(self, first, n):
        """Entries [first, first + n) in the world frame as PointCloud2 float32 xyz records."""
        first, n = self._range(first, n)
        out = np.empty((max(self.rows, 1), 3), dtype=np.float32)
        m = C.c_int64(0)
        self.e._check(self.e.lib.sb_map_world_f32(self.h, first, n, out.ctypes.data_as(C.POINTER(C.c_float)),
                                                  C.byref(m)))
        return out[:m.value].copy()

    def global_map(self, voxel, f32=False):
        """All entries in the world frame, voxel grid at `voxel` (<= 0: the concatenation); float32 records if f32."""
        out = np.empty((max(self.rows, 1), 3), dtype=np.float32 if f32 else np.float64)
        m = C.c_int64(0)
        if f32:
            s = self.e.lib.sb_map_global_f32(self.h, float(voxel), out.ctypes.data_as(C.POINTER(C.c_float)), C.byref(m))
        else:
            s = self.e.lib.sb_map_global(self.h, float(voxel), _dp(out), C.byref(m))
        self.e._check(s)
        return out[:m.value].copy()
