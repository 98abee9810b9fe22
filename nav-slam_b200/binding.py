"""ctypes binding of include/navslam_b200.h -- used by tests, bench.py and smoke().

The product is the C-ABI library (libnavslam_b200.so) and the per-shape reference shims; this
module is only a thin caller.  It FAILS LOUDLY when the CUDA library is missing or no device is
visible: there is no CPU fallback and nothing here imports oracle/.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)
c_i32_p = C.POINTER(C.c_int32)


class NavPos(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("x", "y", "z", "roll", "pitch", "yaw")]


class NavFrameResults(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("labels", "nn_idx", "nn_dist", "global_", "map_mask")]


class NavFrameIO(C.Structure):
    """nav_frame_io of include/navslam_b200.h (pinned host pointers, any output may be None)."""
    _fields_ = [(n, C.c_void_p) for n in ("cloud", "distances", "cloud_out", "feature_out", "mask_out",
                                          "nn_idx_out", "nn_dist_out", "global_out")]


class NavSequenceOut(C.Structure):
    """nav_sequence_out of include/navslam_b200.h (device pointers, any field may be None)."""
    _fields_ = [(n, C.c_void_p) for n in ("label_mask", "nn_idx", "nn_dist", "fit_stats")]


class NavRunDevOut(C.Structure):
    """nav_run_dev_out of include/navslam_b200.h (device pointers; error / fit_stats may be None)."""
    _fields_ = [(n, C.c_void_p) for n in ("poses", "error", "fit_stats")]


class NavError(RuntimeError):
    pass


_LIB = None

# every symbol include/navslam_b200.h declares (tests check the .so exports all of them)
EXPORTS = [
    "nav_version", "nav_last_error", "nav_device_count", "nav_host_alloc", "nav_host_free",
    "nav_create", "nav_destroy", "nav_rows", "nav_cols", "nav_set_stream", "nav_synchronize",
    "nav_launch_count", "nav_convert_to_pointcloud", "nav_extract_feature", "nav_curvature",
    "nav_flatten_points", "nav_transform_cloud", "nav_kdtree_build", "nav_kdtree_build_dev", "nav_kdtree_build_ex",
    "nav_kdtree_free", "nav_kdtree_size", "nav_kdtree_nn_batch", "nav_kdtree_nn_batch_dev",
    "nav_bruteforce_nn_batch_dev", "nav_kdtree_export", "nav_kdtree_launch_count", "nav_slam_init",
    "nav_slam_match", "nav_slam_localization", "nav_slam_mapping", "nav_frontend_frame",
    "nav_extract_feature_batch_dev", "nav_frontend_frame_dev", "nav_slam_init_dev",
    "nav_frame_results_dev", "nav_profile_enable", "nav_profile_read", "nav_row_map_export",
    "nav_exact_fallback_count", "nav_frontend_frame_async", "nav_frontend_wait",
    "nav_frontend_sequence_dev", "nav_slam_localization_fast", "nav_frontend_frame_depth",
    "nav_l9_csv_read", "nav_csv_header", "nav_csv_format_frame", "nav_csv_format_frame_gpu",
    "nav_csv_format_frame_dev", "nav_l5_json_read", "nav_imu_json_read",
    "nav_frontend_submit", "nav_frontend_frame_depth_async", "nav_slam_prefetch", "nav_slam_prefetch_depth",
    "nav_host_register", "nav_host_unregister", "nav_slam_run", "nav_slam_fit_stats",
    "nav_frontend_sequence_out_dev", "nav_slam_fit_from_stats",
    "nav_set_tie_rule", "nav_tie_rule", "nav_tie_resolve_count",
    "nav_peer_create", "nav_peer_connect", "nav_kdtree_nn_allgather_dev", "nav_kdtree_nn_sharded_map_dev", "nav_peer_check",
    "nav_peer_destroy", "nav_shard_range", "nav_shard_owner",
    "nav_frontend_frame_mm", "nav_frontend_submit_mm", "nav_slam_prefetch_mm", "nav_l9_csv_read_mm",
    "nav_slam_run_dev", "nav_slam_init_dev_ex", "nav_frontend_sequence_dev_ex", "nav_slam_run_dev_ex",
]


def lib_path() -> str:
    # NAVSLAM_LIB: developer override (kernel variants built side by side for A/B timing, profiles/prof_frame.py)
    return os.environ.get("NAVSLAM_LIB") or _build.LIB


def load_library(build_if_missing: bool = True):
    """dlopen libnavslam_b200.so (building it with nvcc if it is absent)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        if not build_if_missing:
            raise NavError(f"{path} is missing: run __graft_entry__.build() (needs nvcc)")
        _build.build_library()
    L = C.CDLL(path)
    L.nav_version.restype = C.c_char_p
    L.nav_last_error.restype = C.c_char_p
    L.nav_host_alloc.restype = C.c_void_p
    L.nav_host_alloc.argtypes = [C.c_size_t]
    L.nav_host_free.argtypes = [C.c_void_p]
    L.nav_host_register.argtypes = [C.c_void_p, C.c_size_t]
    L.nav_host_unregister.argtypes = [C.c_void_p]
    L.nav_create.restype = C.c_void_p
    L.nav_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
    L.nav_destroy.argtypes = [C.c_void_p]
    L.nav_rows.argtypes = [C.c_void_p]
    L.nav_cols.argtypes = [C.c_void_p]
    L.nav_set_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    L.nav_synchronize.argtypes = [C.c_void_p]
    L.nav_launch_count.restype = C.c_uint64
    L.nav_launch_count.argtypes = [C.c_void_p]
    vp = C.c_void_p
    L.nav_convert_to_pointcloud.argtypes = [vp, vp, vp]
    L.nav_extract_feature.argtypes = [vp, vp, vp]
    L.nav_curvature.argtypes = [vp, vp, vp]
    L.nav_flatten_points.argtypes = [vp, vp, vp, vp, C.POINTER(C.c_size_t)]
    L.nav_transform_cloud.argtypes = [vp, vp, C.POINTER(NavPos), vp]
    L.nav_kdtree_build.restype = vp
    L.nav_kdtree_build.argtypes = [C.c_int, vp, C.c_size_t]
    L.nav_kdtree_build_dev.restype = vp
    L.nav_kdtree_build_dev.argtypes = [C.c_int, vp, C.c_size_t, vp]
    L.nav_kdtree_free.argtypes = [vp]
    L.nav_kdtree_size.restype = C.c_size_t
    L.nav_kdtree_size.argtypes = [vp]
    L.nav_kdtree_launch_count.restype = C.c_uint64
    L.nav_kdtree_launch_count.argtypes = [vp]
    L.nav_kdtree_nn_batch.argtypes = [vp, vp, C.c_size_t, vp, vp, vp]
    L.nav_kdtree_nn_batch_dev.argtypes = [vp, vp, C.c_size_t, vp, vp, vp]
    L.nav_bruteforce_nn_batch_dev.argtypes = [C.c_int, vp, C.c_size_t, vp, C.c_size_t, vp, vp, C.c_int, vp]
    L.nav_kdtree_export.argtypes = [vp, vp, vp, vp]
    L.nav_kdtree_build_ex.restype = vp
    L.nav_kdtree_build_ex.argtypes = [C.c_int, vp, C.c_size_t, C.c_int, vp, C.c_int]
    L.nav_slam_init.argtypes = [vp, C.POINTER(NavPos), vp, vp]
    L.nav_slam_init_dev.argtypes = [vp, vp, C.POINTER(NavPos)]
    L.nav_slam_match.argtypes = [vp, vp, C.POINTER(NavPos), C.POINTER(NavPos), vp, C.c_size_t,
                                 C.POINTER(C.c_size_t)]
    L.nav_slam_localization.argtypes = [vp, vp, C.POINTER(NavPos), C.POINTER(NavPos), C.POINTER(NavPos),
                                        c_double_p, C.c_int]
    L.nav_slam_localization_fast.argtypes = [vp, vp, C.POINTER(NavPos), C.POINTER(NavPos), C.POINTER(NavPos),
                                             c_double_p, C.POINTER(C.c_size_t)]
    L.nav_slam_mapping.argtypes = [vp, C.POINTER(NavPos), vp, vp]
    L.nav_slam_fit_stats.argtypes = [vp, c_double_p]
    L.nav_slam_fit_from_stats.argtypes = [c_double_p, C.POINTER(NavPos), C.POINTER(NavPos), C.POINTER(NavPos),
                                          c_double_p]
    L.nav_frontend_frame.argtypes = [vp, vp, C.POINTER(NavPos), C.POINTER(NavPos), C.POINTER(NavPos),
                                     vp, vp, vp, vp]
    L.nav_frontend_frame_async.argtypes = [vp, vp, C.POINTER(NavPos), C.POINTER(NavPos), C.POINTER(NavPos),
                                           vp, vp, vp, vp]
    L.nav_frontend_wait.argtypes = [vp]
    L.nav_frontend_submit.argtypes = [vp, C.POINTER(NavFrameIO), C.POINTER(NavPos), C.POINTER(NavPos),
                                      C.POINTER(NavPos)]
    L.nav_frontend_frame_depth_async.argtypes = [vp, vp, C.POINTER(NavPos), C.POINTER(NavPos), C.POINTER(NavPos),
                                                 vp, vp, vp, vp, vp]
    L.nav_slam_run.argtypes = [vp, C.POINTER(C.c_void_p), C.c_int, C.c_int, vp, vp, C.POINTER(NavPos),
                               C.POINTER(NavPos), C.POINTER(NavPos), C.POINTER(C.c_double), C.POINTER(C.c_size_t)]
    L.nav_slam_run_dev.argtypes = [vp, vp, C.c_int, C.POINTER(NavPos), C.POINTER(NavPos), C.POINTER(NavRunDevOut)]
    L.nav_slam_init_dev_ex.argtypes = [vp, vp, C.c_int, C.POINTER(NavPos)]
    L.nav_frontend_sequence_dev_ex.argtypes = [vp, vp, C.c_int, C.c_size_t, C.POINTER(NavPos), C.POINTER(NavPos),
                                               C.POINTER(NavPos), C.POINTER(NavSequenceOut)]
    L.nav_slam_run_dev_ex.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(NavPos), C.POINTER(NavPos),
                                      C.POINTER(NavRunDevOut)]
    L.nav_peer_create.restype = C.c_void_p
    L.nav_peer_create.argtypes = [C.c_int, C.c_size_t, C.c_char_p]
    L.nav_peer_connect.argtypes = [vp, C.c_int, C.c_int, C.c_char_p]
    L.nav_kdtree_nn_allgather_dev.argtypes = [vp, vp, vp, C.c_size_t, C.c_size_t, C.POINTER(C.c_void_p),
                                              C.POINTER(C.c_void_p), vp]
    L.nav_kdtree_nn_sharded_map_dev.argtypes = [vp, vp, vp, C.c_size_t, C.c_int64, C.POINTER(C.c_void_p),
                                                C.POINTER(C.c_void_p), vp]
    L.nav_shard_range.restype = None
    L.nav_shard_range.argtypes = [C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.nav_shard_owner.argtypes = [C.c_int64, C.c_int, C.c_int64]
    L.nav_peer_check.argtypes = [vp]
    L.nav_peer_destroy.argtypes = [vp]
    L.nav_slam_prefetch.argtypes = [vp, vp]
    L.nav_slam_prefetch_depth.argtypes = [vp, vp]
    L.nav_slam_prefetch_mm.argtypes = [vp, vp]
    L.nav_frontend_frame_mm.argtypes = [vp, vp, C.POINTER(NavPos), C.POINTER(NavPos), C.POINTER(NavPos),
                                        vp, vp, vp, vp]
    L.nav_frontend_submit_mm.argtypes = [vp, vp, C.POINTER(NavFrameIO), C.POINTER(NavPos), C.POINTER(NavPos),
                                         C.POINTER(NavPos)]
    L.nav_l9_csv_read_mm.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_size_t, vp, vp, C.POINTER(C.c_size_t)]
    L.nav_l9_csv_read.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_size_t, vp, vp, C.POINTER(C.c_size_t)]
    L.nav_csv_format_frame_gpu.argtypes = [vp, C.c_ulonglong, vp, vp, vp, C.POINTER(NavPos), C.POINTER(NavPos), vp,
                                           C.c_size_t, C.POINTER(C.c_size_t)]
    L.nav_csv_format_frame_dev.argtypes = L.nav_csv_format_frame_gpu.argtypes
    L.nav_l5_json_read.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_size_t, vp, vp, C.POINTER(C.c_size_t)]
    L.nav_imu_json_read.argtypes = [C.c_char_p, C.c_size_t, vp, vp, C.POINTER(C.c_size_t)]
    L.nav_csv_header.restype = C.c_char_p
    L.nav_csv_format_frame.restype = C.c_size_t
    L.nav_csv_format_frame.argtypes = [vp, C.c_size_t, C.c_ulonglong, C.c_int, C.c_int, vp, vp, vp,
                                       C.POINTER(NavPos), C.POINTER(NavPos)]
    L.nav_frontend_frame_depth.argtypes = [vp, vp, C.POINTER(NavPos), C.POINTER(NavPos), C.POINTER(NavPos),
                                           vp, vp, vp, vp, vp]
    L.nav_extract_feature_batch_dev.argtypes = [vp, vp, C.c_size_t, vp]
    L.nav_frontend_frame_dev.argtypes = [vp, vp, C.POINTER(NavPos), C.POINTER(NavPos), C.POINTER(NavPos)]
    L.nav_frontend_sequence_dev.argtypes = [vp, vp, C.c_size_t, C.POINTER(NavPos), C.POINTER(NavPos),
                                            C.POINTER(NavPos)]
    L.nav_frontend_sequence_out_dev.argtypes = [vp, vp, C.c_size_t, C.POINTER(NavPos), C.POINTER(NavPos),
                                                C.POINTER(NavPos), C.POINTER(NavSequenceOut)]
    L.nav_frame_results_dev.argtypes = [vp, C.POINTER(NavFrameResults)]
    L.nav_row_map_export.argtypes = [vp, C.c_int, C.c_int, vp, vp, C.POINTER(C.c_size_t)]
    L.nav_exact_fallback_count.restype = C.c_uint64
    L.nav_exact_fallback_count.argtypes = [vp]
    L.nav_set_tie_rule.argtypes = [vp, C.c_int]
    L.nav_tie_rule.argtypes = [vp]
    L.nav_tie_resolve_count.restype = C.c_uint64
    L.nav_tie_resolve_count.argtypes = [vp]
    L.nav_profile_enable.argtypes = [vp, C.c_int]
    L.nav_profile_read.argtypes = [vp, C.c_char_p, c_double_p, C.POINTER(C.c_uint64), C.c_int]
    _LIB = L
    return L


def _check(rc, L):
    if rc != 0:
        raise NavError(L.nav_last_error().decode("utf-8", "replace"))


def _pos_array(p, n=1):
    """nav_pos[n] from an (n,6) / (6,) array-like."""
    a = np.ascontiguousarray(p, dtype=np.float64).reshape(-1, 6)
    assert a.shape[0] == n, (a.shape, n)
    arr = (NavPos * n)()
    for i in range(n):
        arr[i] = NavPos(*[float(v) for v in a[i]])
    return arr


def _pts(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    assert a.shape[-1] == 3
    return a


def _mm(a):
    """an integer-mm cloud as the C ABI takes it: C-contiguous int32 [..., 3] (no implicit conversion: see to_mm)"""
    if not isinstance(a, np.ndarray) or a.dtype != np.int32:
        raise TypeError("integer-mm clouds are int32 arrays; convert with to_mm()")
    assert a.shape[-1] == 3
    return np.ascontiguousarray(a)


def to_mm(cloud) -> np.ndarray:
    """int32 copy of an xyz cloud in whole millimetres, for the *_mm calls.  Raises ValueError unless every value v
    comes back bit for bit as float64(int32(v)) -- the rule of nav_l9_csv_read_mm: fractions, |v| > 2^31-1, inf, nan
    and -0.0 (whose int32 widens to +0.0) are refused."""
    a = np.ascontiguousarray(cloud, dtype=np.float64)
    in_range = (a >= -2.0 ** 31) & (a <= 2.0 ** 31 - 1)  # False for nan
    m = np.where(in_range, a, 0.0).astype(np.int32)
    bad = ~in_range | (m.astype(np.float64).view(np.uint64) != a.view(np.uint64))
    if bad.any():
        i = np.unravel_index(int(np.argmax(bad)), a.shape)
        raise ValueError(f"to_mm: value {a[i]!r} at index {tuple(int(k) for k in i)} is not a whole number of "
                         f"millimetres that int32 holds with the same float64 bits ({int(bad.sum())} such values)")
    return m


class Context:
    """nav_ctx: one image shape (rows x cols), n_seq sequences side by side, on one device."""

    def __init__(self, rows: int, cols: int, device: int = 0, n_seq: int = 1):
        self.L = load_library()
        self.rows, self.cols, self.n_seq, self.device = rows, cols, n_seq, device
        self.h = self.L.nav_create(rows, cols, device, n_seq)
        if not self.h:
            raise NavError(self.L.nav_last_error().decode("utf-8", "replace"))

    def close(self):
        if getattr(self, "h", None):
            self.L.nav_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    # ---- function level (host buffers)
    def convert_to_pointcloud(self, distances):
        d = np.ascontiguousarray(distances, dtype=np.int32).reshape(self.rows, self.cols)
        out = np.empty((self.rows, self.cols, 3))
        _check(self.L.nav_convert_to_pointcloud(self.h, d.ctypes.data, out.ctypes.data), self.L)
        return out

    def extract_feature(self, cloud, feature=None):
        cloud = _pts(cloud)
        if feature is None:
            feature = np.zeros((self.rows, self.cols), dtype=np.int32)
        assert feature.dtype == np.int32 and feature.flags.c_contiguous
        _check(self.L.nav_extract_feature(self.h, cloud.ctypes.data, feature.ctypes.data), self.L)
        return feature

    def curvature(self, cloud):
        cloud = _pts(cloud)
        out = np.empty((self.rows, self.cols))
        _check(self.L.nav_curvature(self.h, cloud.ctypes.data, out.ctypes.data), self.L)
        return out

    def flatten_points(self, row_points, row_feature):
        row_points = _pts(row_points)
        feat = np.ascontiguousarray(row_feature, dtype=np.int32)
        out = np.empty_like(row_points)
        n = C.c_size_t(0)
        _check(self.L.nav_flatten_points(self.h, row_points.ctypes.data, feat.ctypes.data, out.ctypes.data,
                                         C.byref(n)), self.L)
        return out[:n.value].copy()

    def transform_cloud(self, cloud, pos):
        cloud = _pts(cloud)
        out = np.empty_like(cloud)
        _check(self.L.nav_transform_cloud(self.h, cloud.ctypes.data, _pos_array(pos), out.ctypes.data), self.L)
        return out

    # ---- SLAM step (host buffers)
    def slam_init(self, pos, cloud, want_global=True):
        cloud = _pts(cloud)
        g = np.empty_like(cloud) if want_global else None
        _check(self.L.nav_slam_init(self.h, _pos_array(pos, self.n_seq), cloud.ctypes.data,
                                    g.ctypes.data if g is not None else None), self.L)
        return g

    def slam_match(self, cloud, pos_predict, pos_last):
        cloud = _pts(cloud)
        cap = self.rows * self.cols
        corr = np.empty((cap, 7))
        n = C.c_size_t(0)
        _check(self.L.nav_slam_match(self.h, cloud.ctypes.data, _pos_array(pos_predict), _pos_array(pos_last),
                                     corr.ctypes.data, cap, C.byref(n)), self.L)
        return corr[:n.value].copy()

    def slam_localization(self, cloud, pos_predict, pos_last, verbose=False):
        cloud = _pts(cloud)
        out = NavPos()
        err = C.c_double(0)
        _check(self.L.nav_slam_localization(self.h, cloud.ctypes.data, _pos_array(pos_predict),
                                            _pos_array(pos_last), C.byref(out), C.byref(err),
                                            1 if verbose else 0), self.L)
        return np.array([out.x, out.y, out.z, out.roll, out.pitch, out.yaw]), err.value

    def slam_localization_fast(self, cloud, pos_predict, pos_last):
        cloud = _pts(cloud)
        out = NavPos()
        err = C.c_double(0)
        n = C.c_size_t(0)
        _check(self.L.nav_slam_localization_fast(self.h, cloud.ctypes.data, _pos_array(pos_predict),
                                                 _pos_array(pos_last), C.byref(out), C.byref(err), C.byref(n)),
               self.L)
        return np.array([out.x, out.y, out.z, out.roll, out.pitch, out.yaw]), err.value, int(n.value)

    def slam_mapping(self, pos, cloud=None, want_global=True):
        shape = (self.rows, self.cols, 3) if self.n_seq == 1 else (self.n_seq, self.rows, self.cols, 3)
        g = np.empty(shape) if want_global else None
        cp = None
        if cloud is not None:
            cloud = _pts(cloud)
            cp = cloud.ctypes.data
        _check(self.L.nav_slam_mapping(self.h, _pos_array(pos, self.n_seq), cp,
                                       g.ctypes.data if g is not None else None), self.L)
        return g

    def frontend_frame(self, cloud, pos_predict, pos_last, pos_final):
        cloud = _pts(cloud)
        shp = cloud.shape[:-1]
        feat = np.empty(shp, dtype=np.int32)
        idx = np.empty(shp, dtype=np.int32)
        dist = np.empty(shp)
        g = np.empty_like(cloud)
        n = self.n_seq
        _check(self.L.nav_frontend_frame(self.h, cloud.ctypes.data, _pos_array(pos_predict, n),
                                         _pos_array(pos_last, n), _pos_array(pos_final, n), feat.ctypes.data,
                                         idx.ctypes.data, dist.ctypes.data, g.ctypes.data), self.L)
        return feat, idx, dist, g

    def frontend_frame_depth(self, distances, pos_predict, pos_last, pos_final):
        d = np.ascontiguousarray(distances, dtype=np.int32).reshape(self.rows, self.cols)
        shp = (self.rows, self.cols)
        cloud = np.empty(shp + (3,))
        feat = np.empty(shp, dtype=np.int32)
        idx = np.empty(shp, dtype=np.int32)
        dist = np.empty(shp)
        g = np.empty(shp + (3,))
        _check(self.L.nav_frontend_frame_depth(self.h, d.ctypes.data, _pos_array(pos_predict), _pos_array(pos_last),
                                               _pos_array(pos_final), cloud.ctypes.data, feat.ctypes.data,
                                               idx.ctypes.data, dist.ctypes.data, g.ctypes.data), self.L)
        return cloud, feat, idx, dist, g

    def frontend_frame_mm(self, cloud_mm, pos_predict, pos_last, pos_final):
        """nav_frontend_frame_mm: cloud_mm int32 [..., rows, cols, 3]; returns (labels, nn_idx, nn_dist, global)."""
        m = _mm(cloud_mm)
        shp = m.shape[:-1]
        feat = np.empty(shp, dtype=np.int32)
        idx = np.empty(shp, dtype=np.int32)
        dist = np.empty(shp)
        g = np.empty(shp + (3,))
        n = self.n_seq
        _check(self.L.nav_frontend_frame_mm(self.h, m.ctypes.data, _pos_array(pos_predict, n),
                                            _pos_array(pos_last, n), _pos_array(pos_final, n), feat.ctypes.data,
                                            idx.ctypes.data, dist.ctypes.data, g.ctypes.data), self.L)
        return feat, idx, dist, g

    def csv_rows(self, timestamp, lidar_pos, global_cloud=None, distances=None, imu=None, ekf_pos=None,
                 out_ptr=None, out_cap=0) -> bytes:
        """nav_csv_format_frame_gpu: the frame's CSV lines (src/main.c:320-352) formatted on the GPU.
        global_cloud None = the resident global cloud of the frame mapped last.  out_ptr/out_cap: a pinned
        host buffer to receive the text (then the return value is the byte count)."""
        g = _pts(global_cloud) if global_cloud is not None else None
        d = np.ascontiguousarray(distances, dtype=np.int32) if distances is not None else None
        im = np.ascontiguousarray(imu, dtype=np.float64) if imu is not None else None
        n = C.c_size_t(0)
        if out_ptr is None:
            cap = self.rows * self.cols * 700 + 1024
            buf = C.create_string_buffer(cap)
            ptr = C.addressof(buf)
        else:
            ptr, cap = out_ptr, out_cap
        _check(self.L.nav_csv_format_frame_gpu(self.h, int(timestamp), g.ctypes.data if g is not None else None,
                                               d.ctypes.data if d is not None else None,
                                               im.ctypes.data if im is not None else None, _pos_array(lidar_pos),
                                               _pos_array(ekf_pos) if ekf_pos is not None else None, ptr, cap,
                                               C.byref(n)), self.L)
        return buf.raw[:n.value] if out_ptr is None else n.value

    def frontend_frame_async(self, cloud_ptr, pos_predict, pos_last, pos_final, feat_ptr, idx_ptr, dist_ptr,
                             global_ptr):
        """Pinned host pointers (ints); see nav_frontend_frame_async."""
        n = self.n_seq
        _check(self.L.nav_frontend_frame_async(self.h, cloud_ptr, _pos_array(pos_predict, n),
                                               _pos_array(pos_last, n), _pos_array(pos_final, n), feat_ptr,
                                               idx_ptr, dist_ptr, global_ptr), self.L)

    def frontend_submit(self, pos_predict, pos_last, pos_final, **ptrs):
        """nav_frontend_submit: keyword arguments are the fields of nav_frame_io (pinned host pointers as ints)."""
        io = NavFrameIO(**ptrs)
        n = self.n_seq
        _check(self.L.nav_frontend_submit(self.h, C.byref(io), _pos_array(pos_predict, n), _pos_array(pos_last, n),
                                          _pos_array(pos_final, n)), self.L)

    def frontend_submit_mm(self, cloud_mm_ptr, pos_predict, pos_last, pos_final, **outputs):
        """nav_frontend_submit_mm: cloud_mm_ptr is a pinned int32 [..., 3] frame (int); keyword arguments are the
        output fields of nav_frame_io (pinned host pointers as ints)."""
        io = NavFrameIO(**outputs)
        n = self.n_seq
        _check(self.L.nav_frontend_submit_mm(self.h, cloud_mm_ptr, C.byref(io), _pos_array(pos_predict, n),
                                             _pos_array(pos_last, n), _pos_array(pos_final, n)), self.L)

    def slam_prefetch(self, cloud_ptr=None, depth_ptr=None, mm_ptr=None):
        """nav_slam_prefetch / nav_slam_prefetch_depth / nav_slam_prefetch_mm with a pinned host pointer (int)."""
        if mm_ptr is not None:
            _check(self.L.nav_slam_prefetch_mm(self.h, mm_ptr), self.L)
        elif depth_ptr is not None:
            _check(self.L.nav_slam_prefetch_depth(self.h, depth_ptr), self.L)
        else:
            _check(self.L.nav_slam_prefetch(self.h, cloud_ptr), self.L)

    def slam_localization_fast_ptr(self, cloud_ptr, pos_predict, pos_last):
        """nav_slam_localization_fast on a raw host pointer (int) or None = the oldest prefetched frame."""
        out = NavPos()
        err = C.c_double(0)
        n = C.c_size_t(0)
        _check(self.L.nav_slam_localization_fast(self.h, cloud_ptr, _pos_array(pos_predict), _pos_array(pos_last),
                                                 C.byref(out), C.byref(err), C.byref(n)), self.L)
        return np.array([out.x, out.y, out.z, out.roll, out.pitch, out.yaw]), err.value, int(n.value)

    def slam_fit_stats(self):
        """nav_slam_fit_stats: [N, sum rx, sum ry, sum rz, sum |r|^2] of the last closed-loop fit."""
        out = (C.c_double * 5)()
        _check(self.L.nav_slam_fit_stats(self.h, out), self.L)
        return np.array(out[:])

    RUN_INPUT_XYZ, RUN_INPUT_DEPTH, RUN_INPUT_MM = 0, 1, 2  # NAV_RUN_INPUT_* of include/navslam_b200.h

    def _input_kind(self, name, depth_input, mm_input):
        if depth_input and mm_input:
            raise ValueError(f"{name}: depth_input and mm_input exclude each other")
        return self.RUN_INPUT_DEPTH if depth_input else self.RUN_INPUT_MM if mm_input else self.RUN_INPUT_XYZ

    def slam_run(self, frame_ptrs, deltas, pos_start, depth_input=False, mm_input=False):
        """nav_slam_run: the closed loop over pinned host frames (raw pointers) with dead-reckoning increments
        deltas[t] (prediction = last pose + deltas[t]).  Frames are clouds, depth matrices (depth_input) or int32
        integer-mm clouds (mm_input).  Returns (poses [n,6], rms [n], n_corr [n])."""
        kind = self._input_kind("slam_run", depth_input, mm_input)
        n = len(frame_ptrs)
        ptrs = (C.c_void_p * n)(*[int(p) for p in frame_ptrs])
        d = (NavPos * n)(*[NavPos(*[float(v) for v in row]) for row in np.asarray(deltas, dtype=np.float64).reshape(n, 6)])
        out = (NavPos * n)()
        err = (C.c_double * n)()
        nc = (C.c_size_t * n)()
        _check(self.L.nav_slam_run(self.h, ptrs, n, kind, None, None, d, _pos_array(pos_start),
                                   out, err, nc), self.L)
        poses = np.array([[p.x, p.y, p.z, p.roll, p.pitch, p.yaw] for p in out]).reshape(n, 6)
        return poses, np.array(err[:]), np.array(nc[:], dtype=np.int64)

    def frontend_wait(self):
        _check(self.L.nav_frontend_wait(self.h), self.L)

    # ---- device resident (raw device pointers, e.g. torch tensor .data_ptr())
    def set_stream(self, cuda_stream_handle):
        """Run on the caller's cudaStream_t (0 = legacy default stream); None = the context's own stream."""
        if cuda_stream_handle is None:
            _check(self.L.nav_set_stream(self.h, None, 1), self.L)
        else:
            _check(self.L.nav_set_stream(self.h, cuda_stream_handle, 0), self.L)

    def synchronize(self):
        _check(self.L.nav_synchronize(self.h), self.L)

    def extract_feature_batch_dev(self, dev_clouds_ptr, n_images, dev_labels_ptr):
        _check(self.L.nav_extract_feature_batch_dev(self.h, dev_clouds_ptr, n_images, dev_labels_ptr), self.L)

    def slam_init_dev(self, dev_cloud_ptr, pos, depth_input=False, mm_input=False):
        """nav_slam_init_dev_ex: the map of one device-resident frame -- an xyz cloud, int32 depth matrices
        (depth_input) or an int32 integer-mm cloud (mm_input)."""
        kind = self._input_kind("slam_init_dev", depth_input, mm_input)
        pos = _pos_array(pos, self.n_seq)
        if kind == self.RUN_INPUT_XYZ:
            _check(self.L.nav_slam_init_dev(self.h, dev_cloud_ptr, pos), self.L)
        else:
            _check(self.L.nav_slam_init_dev_ex(self.h, dev_cloud_ptr, kind, pos), self.L)

    def frontend_frame_dev(self, dev_cloud_ptr, pos_predict, pos_last, pos_final):
        n = self.n_seq
        _check(self.L.nav_frontend_frame_dev(self.h, dev_cloud_ptr, _pos_array(pos_predict, n),
                                             _pos_array(pos_last, n), _pos_array(pos_final, n)), self.L)

    def frontend_sequence_dev(self, dev_frames_ptr, n_frames, pos_predict, pos_last, pos_final, depth_input=False,
                              mm_input=False):
        """nav_frontend_sequence_dev[_ex] (out = NULL): the replay of n_frames device-resident frames -- xyz clouds,
        int32 depth matrices (depth_input) or int32 integer-mm clouds (mm_input)."""
        kind = self._input_kind("frontend_sequence_dev", depth_input, mm_input)
        n = n_frames * self.n_seq
        poses = (_pos_array(pos_predict, n), _pos_array(pos_last, n), _pos_array(pos_final, n))
        if kind == self.RUN_INPUT_XYZ:
            _check(self.L.nav_frontend_sequence_dev(self.h, dev_frames_ptr, n_frames, *poses), self.L)
        else:
            _check(self.L.nav_frontend_sequence_dev_ex(self.h, dev_frames_ptr, kind, n_frames, *poses, None), self.L)

    def frontend_sequence_out_dev(self, dev_frames_ptr, n_frames, pos_predict, pos_last, pos_final, label_mask=None,
                                  nn_idx=None, nn_dist=None, fit_stats=None, depth_input=False, mm_input=False):
        """nav_frontend_sequence_out_dev / nav_frontend_sequence_dev_ex: the replay of frontend_sequence_dev keeping
        every frame's results in the given device buffers (ints; None = not wanted).  With all four None the call
        passes out = NULL."""
        kind = self._input_kind("frontend_sequence_out_dev", depth_input, mm_input)
        n = n_frames * self.n_seq
        fields = (label_mask, nn_idx, nn_dist, fit_stats)
        out = None if all(v is None for v in fields) else C.byref(NavSequenceOut(*fields))
        poses = (_pos_array(pos_predict, n), _pos_array(pos_last, n), _pos_array(pos_final, n))
        if kind == self.RUN_INPUT_XYZ:
            _check(self.L.nav_frontend_sequence_out_dev(self.h, dev_frames_ptr, n_frames, *poses, out), self.L)
        else:
            _check(self.L.nav_frontend_sequence_dev_ex(self.h, dev_frames_ptr, kind, n_frames, *poses, out), self.L)

    def slam_run_dev(self, dev_frames_ptr, n_frames, deltas, pos_start, poses_ptr, error_ptr=None, stats_ptr=None,
                     depth_input=False, mm_input=False):
        """nav_slam_run_dev_ex: the closed loop over n_frames device-resident frames [n_frames][n_seq][rows][cols] --
        xyz clouds, int32 depth matrices (depth_input) or int32 integer-mm clouds (mm_input) -- with the pose fit on
        the GPU.  deltas [n_frames][n_seq][6] (prediction = last pose + deltas[t]), pos_start [n_seq][6]; the outputs
        are device buffers (ints): poses nav_pos [n_frames][n_seq], error double [n_frames][n_seq] and stats double
        [n_frames][n_seq][5] (None = not wanted).  Queued on the context's stream; the outputs are complete after
        synchronize()."""
        kind = self._input_kind("slam_run_dev", depth_input, mm_input)
        n = n_frames * self.n_seq
        d = _pos_array(deltas, n) if n > 0 else (NavPos * 1)()
        out = NavRunDevOut(poses_ptr, error_ptr, stats_ptr)
        start = _pos_array(pos_start, self.n_seq)
        if kind == self.RUN_INPUT_XYZ:
            _check(self.L.nav_slam_run_dev(self.h, dev_frames_ptr, n_frames, d, start, C.byref(out)), self.L)
        else:
            _check(self.L.nav_slam_run_dev_ex(self.h, dev_frames_ptr, kind, n_frames, d, start, C.byref(out)), self.L)

    def frame_results_dev(self) -> NavFrameResults:
        r = NavFrameResults()
        _check(self.L.nav_frame_results_dev(self.h, C.byref(r)), self.L)
        return r

    def row_map_export(self, row, seq=0):
        pts = np.empty((self.cols, 3))
        col = np.empty(self.cols, dtype=np.int32)
        n = C.c_size_t(0)
        _check(self.L.nav_row_map_export(self.h, seq, row, pts.ctypes.data, col.ctypes.data, C.byref(n)), self.L)
        return pts[:n.value].copy(), col[:n.value].copy()

    def exact_fallback_count(self) -> int:
        return int(self.L.nav_exact_fallback_count(self.h))

    TIE_RULES = {"lowest_index": 0, "reference": 1}  # NAV_TIE_* of include/navslam_b200.h

    def set_tie_rule(self, rule: str):
        """nav_set_tie_rule: "lowest_index" (default) or "reference" (the reference's nearest point on exact
        distance ties; blocking calls only, see include/navslam_b200.h)."""
        if rule not in self.TIE_RULES:
            raise ValueError(f"unknown tie rule {rule!r}; expected one of {sorted(self.TIE_RULES)}")
        _check(self.L.nav_set_tie_rule(self.h, self.TIE_RULES[rule]), self.L)

    @property
    def tie_rule(self) -> str:
        v = int(self.L.nav_tie_rule(self.h))
        return {n: k for k, n in self.TIE_RULES.items()}[v]

    def tie_resolve_count(self) -> int:
        """tied queries re-answered by the host under the "reference" rule since the context was created"""
        return int(self.L.nav_tie_resolve_count(self.h))

    def launch_count(self) -> int:
        return int(self.L.nav_launch_count(self.h))

    def profile_enable(self, on=True):
        _check(self.L.nav_profile_enable(self.h, 1 if on else 0), self.L)

    def profile_read(self, name, reset=False):
        ms = C.c_double(0)
        n = C.c_uint64(0)
        _check(self.L.nav_profile_read(self.h, name.encode(), C.byref(ms), C.byref(n), 1 if reset else 0), self.L)
        return ms.value, int(n.value)


class KdTree:
    """nav_kdtree: flat device-resident kd-tree over n points."""

    SPLIT = {"cyclic": 0, "widest": 1}  # NAV_KD_SPLIT_* of include/navslam_b200.h

    def __init__(self, points=None, device: int = 0, *, dev_ptr=None, n=None, stream=None, split=None):
        """split: None = the library default (widest extent), "cyclic" = depth % 3 like utils/kdtree.c:72."""
        self.L = load_library()
        self.device = device
        if dev_ptr is not None:
            if split is None:
                self.h = self.L.nav_kdtree_build_dev(device, dev_ptr, n, stream)
            else:
                self.h = self.L.nav_kdtree_build_ex(device, dev_ptr, n, 1, stream, self.SPLIT[split])
        else:
            pts = _pts(points)
            self._n = pts.shape[0]
            if split is None:
                self.h = self.L.nav_kdtree_build(device, pts.ctypes.data, pts.shape[0])
            else:
                self.h = self.L.nav_kdtree_build_ex(device, pts.ctypes.data, pts.shape[0], 0, None, self.SPLIT[split])
        if not self.h:
            raise NavError(self.L.nav_last_error().decode("utf-8", "replace"))

    def close(self):
        if getattr(self, "h", None):
            self.L.nav_kdtree_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def __len__(self):
        return int(self.L.nav_kdtree_size(self.h))

    def nn_batch(self, queries, want_nearest=True):
        q = _pts(queries)
        nq = q.shape[0]
        idx = np.empty(nq, dtype=np.int32)
        dist = np.empty(nq)
        near = np.full((nq, 3), np.nan) if want_nearest else None
        _check(self.L.nav_kdtree_nn_batch(self.h, q.ctypes.data, nq, idx.ctypes.data, dist.ctypes.data,
                                          near.ctypes.data if near is not None else None), self.L)
        return idx, dist, near

    def nn_batch_dev(self, dev_q_ptr, nq, dev_idx_ptr, dev_dist_ptr, stream=None):
        _check(self.L.nav_kdtree_nn_batch_dev(self.h, dev_q_ptr, nq, dev_idx_ptr, dev_dist_ptr, stream), self.L)

    def export(self, with_axes=False):
        n = len(self)
        nodes = np.empty((n, 3))
        idx = np.empty(n, dtype=np.int32)
        axes = np.empty(n, dtype=np.int32)
        _check(self.L.nav_kdtree_export(self.h, nodes.ctypes.data, idx.ctypes.data, axes.ctypes.data), self.L)
        return (nodes, idx, axes) if with_axes else (nodes, idx)

    def launch_count(self) -> int:
        return int(self.L.nav_kdtree_launch_count(self.h))


def bruteforce_nn_dev(device, dev_pts_ptr, n, dev_q_ptr, nq, dev_idx_ptr, dev_dist_ptr, use_tensor_cores=False,
                      stream=None):
    L = load_library()
    _check(L.nav_bruteforce_nn_batch_dev(device, dev_pts_ptr, n, dev_q_ptr, nq, dev_idx_ptr, dev_dist_ptr,
                                         1 if use_tensor_cores else 0, stream), L)


def l9_csv_read(path, rows, cols, max_frames):
    """nav_l9_csv_read: returns (frames [n,rows,cols,3] float64, timestamps [n] int32)."""
    L = load_library()
    frames = np.zeros((max_frames, rows, cols, 3))
    ts = np.zeros(max_frames, dtype=np.int32)
    n = C.c_size_t(0)
    _check(L.nav_l9_csv_read(path.encode(), rows, cols, max_frames, frames.ctypes.data, ts.ctypes.data, C.byref(n)), L)
    return frames[:n.value], ts[:n.value]


def l9_csv_read_mm(path, rows, cols, max_frames):
    """nav_l9_csv_read_mm: returns (frames [n,rows,cols,3] int32, timestamps [n] int32); fails on any value that is
    not an exact int32 (see to_mm)."""
    L = load_library()
    frames = np.zeros((max_frames, rows, cols, 3), dtype=np.int32)
    ts = np.zeros(max_frames, dtype=np.int32)
    n = C.c_size_t(0)
    _check(L.nav_l9_csv_read_mm(path.encode(), rows, cols, max_frames, frames.ctypes.data, ts.ctypes.data,
                                C.byref(n)), L)
    return frames[:n.value], ts[:n.value]


def l5_json_read(path, rows, cols, max_frames, fill=0):
    """nav_l5_json_read: returns (distances [n,rows,cols] int32, timestamps [n] int32)."""
    L = load_library()
    d = np.full((max_frames, rows, cols), fill, dtype=np.int32)
    ts = np.zeros(max_frames, dtype=np.int32)
    n = C.c_size_t(0)
    _check(L.nav_l5_json_read(path.encode(), rows, cols, max_frames, d.ctypes.data, ts.ctypes.data, C.byref(n)), L)
    return d[:n.value], ts[:n.value]


def imu_json_read(path, max_frames):
    """nav_imu_json_read: returns (params [n,6] = roll,pitch,yaw,x,y,z, timestamps [n] int32)."""
    L = load_library()
    p = np.zeros((max_frames, 6))
    ts = np.zeros(max_frames, dtype=np.int32)
    n = C.c_size_t(0)
    _check(L.nav_imu_json_read(path.encode(), max_frames, p.ctypes.data, ts.ctypes.data, C.byref(n)), L)
    return p[:n.value], ts[:n.value]


def csv_format_frame(timestamp, global_cloud, lidar_pos, distances=None, imu=None, ekf_pos=None) -> bytes:
    """nav_csv_format_frame: the rows*cols CSV lines of one frame (src/main.c:320-352)."""
    L = load_library()
    g = _pts(global_cloud)
    rows, cols = g.shape[0], g.shape[1]
    buf = C.create_string_buffer(rows * cols * 400 + 1024)
    d = np.ascontiguousarray(distances, dtype=np.int32) if distances is not None else None
    im = np.ascontiguousarray(imu, dtype=np.float64) if imu is not None else None
    n = L.nav_csv_format_frame(buf, len(buf), int(timestamp), rows, cols, g.ctypes.data,
                               d.ctypes.data if d is not None else None, im.ctypes.data if im is not None else None,
                               _pos_array(lidar_pos), _pos_array(ekf_pos) if ekf_pos is not None else None)
    if n == 0:
        raise NavError("nav_csv_format_frame: buffer too small")
    return buf.raw[:n]


def fit_from_stats(stats, pos_predict, pos_last):
    """nav_slam_fit_from_stats: the closed loop's host fit on five totals [N, sum rx, sum ry, sum rz, sum |r|^2].
    Returns (pose [6], rms error)."""
    L = load_library()
    st = (C.c_double * 5)(*[float(v) for v in np.asarray(stats, dtype=np.float64).reshape(5)])
    out = NavPos()
    err = C.c_double(0)
    _check(L.nav_slam_fit_from_stats(st, _pos_array(pos_predict), _pos_array(pos_last), C.byref(out), C.byref(err)), L)
    return np.array([out.x, out.y, out.z, out.roll, out.pitch, out.yaw]), err.value


def device_count() -> int:
    return int(load_library().nav_device_count())
