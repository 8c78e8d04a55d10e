"""Test-side loader for oracle/_ref/libslam_ref.so: the reference's own sources compiled against the Eigen stand-in
(oracle/build_ref.sh, oracle/ref_harness.cpp).  TEST INFRASTRUCTURE ONLY.

The library can only be BUILT from a checkout of the original project (REFERENCE_ROOT names it; its sources are not
part of this repository).  Tests that need it skip when it is absent.
"""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "oracle", "_ref", "libslam_ref.so")

_D = C.POINTER(C.c_double)
_I = C.POINTER(C.c_int)


def _dp(a):
    return a.ctypes.data_as(_D)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64).reshape(-1, 3)


def build():
    """(Re)build when REFERENCE_ROOT names the original project's checkout and the harness or the stand-in is newer
    than the library."""
    root = os.environ.get("REFERENCE_ROOT")
    if not root or not os.path.isdir(os.path.join(root, "slam_viz", "include")):
        return
    srcs = [os.path.join(ROOT, "oracle", "ref_harness.cpp"), os.path.join(ROOT, "oracle", "build_ref.sh"),
            os.path.join(ROOT, "oracle", "eigen_standin", "Eigen", "Dense")]
    if not os.path.exists(SO) or any(os.path.getmtime(s) > os.path.getmtime(SO) for s in srcs):
        subprocess.check_call(["sh", os.path.join(ROOT, "oracle", "build_ref.sh")])


def available():
    build()
    return os.path.exists(SO)


class Reference:
    def __init__(self):
        build()
        lib = C.CDLL(SO)
        lib.ref_voxel_downsample.restype = C.c_longlong
        lib.ref_voxel_downsample.argtypes = [_D, C.c_longlong, C.c_double, _D]
        lib.ref_load_points.restype = C.c_longlong
        lib.ref_load_points.argtypes = [C.c_char_p, C.c_int, _D, C.c_longlong]
        lib.ref_kdtree_build.restype = C.c_void_p
        lib.ref_kdtree_build.argtypes = [_D, C.c_int]
        lib.ref_kdtree_free.argtypes = [C.c_void_p]
        lib.ref_kdtree_nearest_batch.argtypes = [C.c_void_p, _D, C.c_int, _I, _D]
        lib.ref_kdtree_nearest.restype = C.c_int
        lib.ref_kdtree_nearest.argtypes = [C.c_void_p, _D]
        lib.ref_kdtree_k_nearest_batch.argtypes = [C.c_void_p, _D, C.c_int, C.c_int, _I]
        lib.ref_find_correspondences.argtypes = [_D, C.c_int, _D, C.c_int, _D, _D]
        lib.ref_estimate_normals.argtypes = [C.c_void_p, C.c_int, _D]
        lib.ref_solve_point_to_plane.argtypes = [_D, _D, _D, C.c_int, _D]
        lib.ref_icp_point_to_plane.restype = C.c_int
        lib.ref_icp_point_to_plane.argtypes = [_D, C.c_int, _D, C.c_int, C.c_int, C.c_double, C.c_double, _D, _D, _I, _I,
                                               _D, _D]
        lib.ref_transform_apply.argtypes = [_D, _D, C.c_longlong, _D]
        lib.ref_transform_compose_inverse.argtypes = [_D, _D, _D, _D]
        lib.ref_sc_compute.argtypes = [_D, C.c_longlong, _D]
        lib.ref_sc_distance_clouds.restype = C.c_double
        lib.ref_sc_distance_clouds.argtypes = [_D, C.c_longlong, _D, C.c_longlong]
        lib.ref_sc_keys.argtypes = [_D, C.c_longlong, _D, _D]
        lib.ref_loop_create.restype = C.c_void_p
        lib.ref_loop_create.argtypes = [C.c_int, C.c_double, C.c_double, C.c_int]
        lib.ref_loop_free.argtypes = [C.c_void_p]
        lib.ref_loop_add.argtypes = [C.c_void_p, _D, C.c_int, C.c_int]
        lib.ref_loop_size.argtypes = [C.c_void_p]
        lib.ref_loop_clear.argtypes = [C.c_void_p]
        lib.ref_loop_detect.restype = C.c_int
        lib.ref_loop_detect.argtypes = [C.c_void_p, C.c_int, _I, _D, _D, _D]
        self.lib = lib

    def voxel_downsample(self, pts, voxel):
        """Rows in the reference's unordered_map order; callers sort."""
        p = _f64(pts)
        out = np.empty_like(p)
        m = self.lib.ref_voxel_downsample(_dp(p), p.shape[0], voxel, _dp(out))
        return out[:m].copy()

    def load_points(self, path, is_bin, capacity=1 << 22):
        out = np.empty((capacity, 3))
        m = self.lib.ref_load_points(path.encode(), int(is_bin), _dp(out), capacity)
        return out[:m].copy()

    class Tree:
        def __init__(self, lib, pts):
            self.lib = lib
            self.p = _f64(pts)
            self.h = lib.ref_kdtree_build(_dp(self.p), self.p.shape[0])

        def __del__(self):
            if getattr(self, "h", None):
                self.lib.ref_kdtree_free(self.h)
                self.h = None

        def nearest_batch(self, q):
            q = _f64(q)
            idx = np.empty(q.shape[0], dtype=np.int32)
            d2 = np.empty(q.shape[0])
            self.lib.ref_kdtree_nearest_batch(self.h, _dp(q), q.shape[0], idx.ctypes.data_as(_I), _dp(d2))
            return idx, d2

        def nearest(self, q):
            q = np.ascontiguousarray(q, dtype=np.float64).reshape(3)
            return int(self.lib.ref_kdtree_nearest(self.h, _dp(q)))

        def k_nearest_batch(self, q, k):
            q = _f64(q)
            out = np.empty((q.shape[0], k), dtype=np.int32)
            self.lib.ref_kdtree_k_nearest_batch(self.h, _dp(q), q.shape[0], k, out.ctypes.data_as(_I))
            return out

        def estimate_normals(self, k):
            n = np.empty_like(self.p)
            self.lib.ref_estimate_normals(self.h, k, _dp(n))
            return n

    def tree(self, pts):
        return Reference.Tree(self.lib, pts)

    def find_correspondences(self, tgt, src):
        t, s = _f64(tgt), _f64(src)
        m = np.empty_like(s)
        d = np.empty(s.shape[0])
        self.lib.ref_find_correspondences(_dp(t), t.shape[0], _dp(s), s.shape[0], _dp(m), _dp(d))
        return m, d

    def solve_point_to_plane(self, src, tgt, nrm):
        s, t, n = _f64(src), _f64(tgt), _f64(nrm)
        T = np.empty(16)
        self.lib.ref_solve_point_to_plane(_dp(s), _dp(t), _dp(n), s.shape[0], _dp(T))
        return T.reshape(4, 4)

    def icp_point_to_plane(self, src, tgt, max_iterations=50, tolerance=1e-6, min_error=1e-9, T0=None):
        s, t = _f64(src), _f64(tgt)
        T = np.empty(16)
        conv, nit = C.c_int(0), C.c_int(0)
        fe = C.c_double(0)
        hist = np.empty(max_iterations + 2)
        t0 = None if T0 is None else np.ascontiguousarray(T0, dtype=np.float64).reshape(16)
        hl = self.lib.ref_icp_point_to_plane(_dp(s), s.shape[0], _dp(t), t.shape[0], max_iterations, tolerance,
                                             min_error, _dp(t0) if t0 is not None else None, _dp(T), C.byref(conv),
                                             C.byref(nit), C.byref(fe), _dp(hist))
        return dict(transformation=T.reshape(4, 4), converged=bool(conv.value), num_iterations=nit.value,
                    final_error=fe.value, error_history=hist[:hl].copy())

    def transform_apply(self, T, pts):
        p, T = _f64(pts), np.ascontiguousarray(T, dtype=np.float64).reshape(16)
        out = np.empty_like(p)
        self.lib.ref_transform_apply(_dp(T), _dp(p), p.shape[0], _dp(out))
        return out

    def compose_inverse(self, A, B):
        A = np.ascontiguousarray(A, dtype=np.float64).reshape(16)
        B = np.ascontiguousarray(B, dtype=np.float64).reshape(16)
        AB, Ai = np.empty(16), np.empty(16)
        self.lib.ref_transform_compose_inverse(_dp(A), _dp(B), _dp(AB), _dp(Ai))
        return AB.reshape(4, 4), Ai.reshape(4, 4)

    def sc_compute(self, pts):
        p = _f64(pts)
        d = np.empty(1200)
        self.lib.ref_sc_compute(_dp(p), p.shape[0], _dp(d))
        return d

    def sc_distance_clouds(self, a, b):
        a, b = _f64(a), _f64(b)
        return float(self.lib.ref_sc_distance_clouds(_dp(a), a.shape[0], _dp(b), b.shape[0]))

    def sc_keys(self, pts):
        p = _f64(pts)
        r, s = np.empty(20), np.empty(60)
        self.lib.ref_sc_keys(_dp(p), p.shape[0], _dp(r), _dp(s))
        return r, s

    class Loop:
        def __init__(self, lib, frame_gap, sc_thr, icp_thr, max_candidates):
            self.lib = lib
            self.h = lib.ref_loop_create(frame_gap, sc_thr, icp_thr, max_candidates)

        def __del__(self):
            if getattr(self, "h", None):
                self.lib.ref_loop_free(self.h)
                self.h = None

        def add(self, pts, frame_idx):
            p = _f64(pts)
            self.lib.ref_loop_add(self.h, _dp(p), p.shape[0], frame_idx)

        def size(self):
            return int(self.lib.ref_loop_size(self.h))

        def clear(self):
            self.lib.ref_loop_clear(self.h)

        def detect(self, cap=64):
            fr = np.empty(2 * cap, dtype=np.int32)
            T = np.empty(16 * cap)
            sd, fit = np.empty(cap), np.empty(cap)
            m = min(self.lib.ref_loop_detect(self.h, cap, fr.ctypes.data_as(_I), _dp(T), _dp(sd), _dp(fit)), cap)
            return [dict(query_frame=int(fr[2 * i]), match_frame=int(fr[2 * i + 1]),
                         transform=T[16 * i:16 * i + 16].reshape(4, 4).copy(), scan_context_distance=float(sd[i]),
                         icp_fitness=float(fit[i])) for i in range(m)]

    def loop(self, frame_gap=50, sc_thr=0.25, icp_thr=0.3, max_candidates=3):
        return Reference.Loop(self.lib, frame_gap, sc_thr, icp_thr, max_candidates)
