"""ctypes bindings for the two CPU checkers (TEST INFRASTRUCTURE):

  * Oracle  -- oracle/_build/libnavoracle.so, our C restatement (runtime shapes)
  * RefLib  -- oracle/_ref/libnavref_<RxC>.so, the reference's own sources compiled
               per shape by oracle/build_ref.sh (present only if it was built where
               /root/reference exists; it travels to the GPU box as a binary)

Nothing in nav-slam_b200/ imports this module.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import os
import subprocess
from contextlib import contextmanager

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "_build", "libnavoracle.so")
REF_DIR = os.path.join(ORACLE_DIR, "_ref")

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)
c_i32_p = C.POINTER(C.c_int32)


class Pos(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("x", "y", "z", "roll", "pitch", "yaw")]

    @classmethod
    def of(cls, v):
        v = [float(t) for t in v]
        return cls(*v)

    def arr(self):
        return np.array([self.x, self.y, self.z, self.roll, self.pitch, self.yaw])


def _dp(a):
    return a.ctypes.data_as(c_double_p)


def _ip(a):
    return a.ctypes.data_as(c_int_p)


def _pts(a) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.float64)
    assert a.shape[-1] == 3
    return a


def build_oracle():
    if not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(
            os.path.join(ORACLE_DIR, "navslam_oracle.c")):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "oracle"], stdout=subprocess.DEVNULL)
    return ORACLE_SO


@contextmanager
def quiet_stdout():
    """The reference prints every Adam iteration (src/slam.c:372); silence fd 1 around it."""
    import sys
    sys.stdout.flush()
    saved = os.dup(1)
    devnull = os.open(os.devnull, os.O_WRONLY)
    try:
        os.dup2(devnull, 1)
        yield
    finally:
        C.CDLL(None).fflush(None)
        os.dup2(saved, 1)
        os.close(saved)
        os.close(devnull)


class Oracle:
    def __init__(self):
        self.lib = C.CDLL(build_oracle())
        L = self.lib
        L.nso_flatten.restype = C.c_size_t
        L.nso_tree_build.restype = C.c_void_p
        L.nso_tree_build.argtypes = [c_double_p, C.c_size_t, C.c_int]
        L.nso_tree_free.argtypes = [C.c_void_p]
        L.nso_tree_nn.argtypes = [C.c_void_p, c_double_p, c_double_p, c_double_p, C.c_int]
        L.nso_tree_preorder.restype = C.c_size_t
        L.nso_tree_preorder.argtypes = [C.c_void_p, c_double_p, c_int_p, C.c_size_t]
        L.nso_nn_brute.argtypes = [c_double_p, C.c_size_t, c_double_p, C.c_size_t, c_i32_p, c_double_p]
        L.nso_nn_tie_count.argtypes = [c_double_p, C.c_size_t, c_double_p, C.c_size_t, c_i32_p]
        L.nso_slam_create.restype = C.c_void_p
        L.nso_slam_create.argtypes = [C.c_int, C.c_int, C.c_int]
        L.nso_slam_destroy.argtypes = [C.c_void_p]
        L.nso_slam_init.argtypes = [C.c_void_p, C.POINTER(Pos), c_double_p, c_double_p]
        L.nso_slam_map.argtypes = [C.c_void_p, C.POINTER(Pos), c_double_p, c_double_p]
        L.nso_slam_localize.restype = C.c_size_t
        L.nso_slam_localize.argtypes = [C.c_void_p, c_double_p, C.POINTER(Pos), C.POINTER(Pos),
                                        C.POINTER(Pos), c_double_p, C.c_size_t, c_int_p]
        L.nso_slam_error.restype = C.c_double
        L.nso_slam_error.argtypes = [C.c_void_p]
        L.nso_slam_frame_count.argtypes = [C.c_void_p]
        L.nso_frontend_frame.argtypes = [C.c_void_p, c_double_p, C.POINTER(Pos), C.POINTER(Pos),
                                         C.POINTER(Pos), c_int_p, c_i32_p, c_double_p, c_double_p]

        L.nso_l9_csv_read.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p,
                                      C.POINTER(C.c_size_t)]
        L.nso_csv_format_frame.restype = C.c_size_t
        L.nso_csv_format_frame.argtypes = [C.c_void_p, C.c_size_t, C.c_ulonglong, C.c_int, C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.POINTER(Pos), C.POINTER(Pos)]

    # --- caller-side data formats
    def l9_csv_read(self, path, rows, cols, max_frames):
        frames = np.zeros((max_frames, rows, cols, 3))
        ts = np.zeros(max_frames, dtype=np.int32)
        n = C.c_size_t(0)
        rc = self.lib.nso_l9_csv_read(path.encode(), rows, cols, max_frames, frames.ctypes.data, ts.ctypes.data,
                                      C.byref(n))
        return rc, frames[:n.value], ts[:n.value]

    def csv_format_frame(self, timestamp, g, lidar_pos, distances=None, imu=None, ekf_pos=None) -> bytes:
        g = _pts(g)
        rows, cols = g.shape[0], g.shape[1]
        buf = C.create_string_buffer(rows * cols * 25 * 330 + 1024)
        d = np.ascontiguousarray(distances, dtype=np.int32) if distances is not None else None
        im = np.ascontiguousarray(imu, dtype=np.float64) if imu is not None else None
        lp = Pos.of(lidar_pos)
        ep = Pos.of(ekf_pos) if ekf_pos is not None else None
        n = self.lib.nso_csv_format_frame(buf, len(buf), int(timestamp), rows, cols, g.ctypes.data,
                                          d.ctypes.data if d is not None else None,
                                          im.ctypes.data if im is not None else None, C.byref(lp),
                                          C.byref(ep) if ep is not None else None)
        assert n > 0
        return buf.raw[:n]

    # --- function level
    def convert(self, dist):
        dist = np.ascontiguousarray(dist, dtype=np.int32)
        r, c = dist.shape
        out = np.empty((r, c, 3))
        self.lib.nso_convert_to_pointcloud(r, c, _ip(dist), _dp(out))
        return out

    def curvature(self, cloud):
        cloud = _pts(cloud)
        r, c, _ = cloud.shape
        out = np.empty((r, c))
        self.lib.nso_curvature(r, c, _dp(cloud), _dp(out))
        return out

    def extract_feature(self, cloud, feature=None):
        cloud = _pts(cloud)
        r, c, _ = cloud.shape
        if feature is None:
            feature = np.zeros((r, c), dtype=np.int32)
        self.lib.nso_extract_feature(r, c, _dp(cloud), _ip(feature))
        return feature

    def flatten(self, row, feat):
        row = _pts(row)
        feat = np.ascontiguousarray(feat, dtype=np.int32)
        out = np.empty_like(row)
        n = self.lib.nso_flatten(row.shape[0], _dp(row), _ip(feat), _dp(out))
        return out[:n].copy()

    def rotation_deg(self, pos):
        R = np.empty(9)
        p = Pos.of(pos)
        self.lib.nso_deg_rotation(C.byref(p), _dp(R))
        return R

    def transform(self, pts, pos):
        pts = _pts(pts)
        R = self.rotation_deg(pos)
        t = np.array(pos[:3], dtype=np.float64)
        out = np.empty_like(pts)
        self.lib.nso_transform(C.c_size_t(pts.size // 3), _dp(pts), _dp(R), _dp(t), _dp(out))
        return out

    def shift(self, pts, d):
        pts = _pts(pts)
        d = np.ascontiguousarray(d, dtype=np.float64)
        out = np.empty_like(pts)
        self.lib.nso_shift(C.c_size_t(pts.size // 3), _dp(pts), _dp(d), _dp(out))
        return out

    def tree_build(self, pts):
        """Returns (handle, permuted copy).  Reference-shaped tree (Lomuto quick-select)."""
        work = _pts(pts).copy()
        h = self.lib.nso_tree_build(_dp(work), work.shape[0], 0)
        return h, work

    def tree_free(self, h):
        self.lib.nso_tree_free(h)

    def tree_nn(self, h, q):
        q = _pts(q)
        out = np.full_like(q, np.nan)
        dist = np.full(q.shape[0], np.inf)
        for i in range(q.shape[0]):
            self.lib.nso_tree_nn(h, _dp(q[i:i + 1]), _dp(out[i:i + 1]), _dp(dist[i:i + 1]), 0)
        return out, dist

    def tree_preorder(self, h, n):
        out = np.empty((n, 3))
        depth = np.empty(n, dtype=np.int32)
        k = self.lib.nso_tree_preorder(h, _dp(out), _ip(depth), n)
        return out[:k], depth[:k]

    def nn_brute(self, pts, q):
        pts, q = _pts(pts), _pts(q)
        idx = np.empty(q.shape[0], dtype=np.int32)
        dist = np.empty(q.shape[0])
        self.lib.nso_nn_brute(_dp(pts), pts.shape[0], _dp(q), q.shape[0],
                              idx.ctypes.data_as(c_i32_p), _dp(dist))
        return idx, dist

    def nn_tie_count(self, pts, q):
        pts, q = _pts(pts), _pts(q)
        cnt = np.empty(q.shape[0], dtype=np.int32)
        self.lib.nso_nn_tie_count(_dp(pts), pts.shape[0], _dp(q), q.shape[0], cnt.ctypes.data_as(c_i32_p))
        return cnt

    # --- whole step
    def slam(self, rows, cols, tie_mode):
        return OracleSlam(self, rows, cols, tie_mode)


class OracleSlam:
    def __init__(self, oracle: Oracle, rows, cols, tie_mode):
        self.o, self.rows, self.cols = oracle, rows, cols
        self.h = oracle.lib.nso_slam_create(rows, cols, tie_mode)

    def close(self):
        if self.h:
            self.o.lib.nso_slam_destroy(self.h)
            self.h = None

    __del__ = close

    def init(self, pos, cloud):
        cloud = _pts(cloud)
        g = np.empty_like(cloud)
        p = Pos.of(pos)
        self.o.lib.nso_slam_init(self.h, C.byref(p), _dp(cloud), _dp(g))
        return g

    def map(self, pos, cloud):
        cloud = _pts(cloud)
        g = np.empty_like(cloud)
        p = Pos.of(pos)
        self.o.lib.nso_slam_map(self.h, C.byref(p), _dp(cloud), _dp(g))
        return g

    def localize(self, cloud, pos_predict, pos_last):
        cloud = _pts(cloud)
        cap = self.rows * self.cols
        corr = np.empty((cap, 7))
        out = Pos()
        iters = C.c_int(0)
        pp, pl = Pos.of(pos_predict), Pos.of(pos_last)
        n = self.o.lib.nso_slam_localize(self.h, _dp(cloud), C.byref(pp), C.byref(pl), C.byref(out),
                                         _dp(corr), cap, C.byref(iters))
        return out.arr(), corr[:n].copy(), self.o.lib.nso_slam_error(self.h), iters.value

    def frontend_frame(self, cloud, pos_predict, pos_last, pos_final):
        cloud = _pts(cloud)
        n = self.rows * self.cols
        feat = np.empty((self.rows, self.cols), dtype=np.int32)
        idx = np.empty(n, dtype=np.int32)
        dist = np.empty(n)
        g = np.empty_like(cloud)
        pp, pl, pf = Pos.of(pos_predict), Pos.of(pos_last), Pos.of(pos_final)
        self.o.lib.nso_frontend_frame(self.h, _dp(cloud), C.byref(pp), C.byref(pl), C.byref(pf),
                                      _ip(feat), idx.ctypes.data_as(c_i32_p), _dp(dist), _dp(g))
        return feat, idx.reshape(self.rows, self.cols), dist.reshape(self.rows, self.cols), g


def ref_available(shape: str) -> bool:
    return os.path.exists(os.path.join(REF_DIR, f"libnavref_{shape}.so"))


# ------------------------------------------------------------------ stored reference answers
# The reference's sources are not part of this repository, so oracle/_ref is usually absent.  Every
# comparison with it goes through check_ref(): against RefLib where oracle/_ref is built, otherwise against
# the sha256 digest of the same answer stored in tests/golden/ref_digests.json.  Where oracle/_ref is built,
# check_ref() also holds the stored digest to the live answer, so every such run validates the file.  The
# file says what its answers were recorded from ("recorded_from") and lists the keys that were never
# compared with the reference ("never_compared_with_the_reference"); tests/test_golden.py ties the keys it
# shares with the reference-generated tests/golden/ref_*.npz to those vectors.
# tests/golden/make_ref_digests.py re-records the file.
REF_DIGESTS = os.path.join(ROOT, "tests", "golden", "ref_digests.json")
_RECORD_TO = os.environ.get("NAVSLAM_RECORD_REF_DIGESTS")
_digests = None
_recorded = {}


def digest(a) -> str:
    """sha256 over dtype, shape and bytes: equal digests mean bit-identical arrays."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def stored_answers() -> dict:
    global _digests
    if _digests is None:
        with open(REF_DIGESTS) as f:
            _digests = json.load(f)["answers"]
    return _digests


def check_ref(key: str, got, ref_fn=None, also=()):
    """Assert that `got` is bit-identical to the reference's answer for `key`: ref_fn() (the live reference)
    when it is given, else the stored digest.  `also` lists other forms of our answer that the reference may
    equally give (the first one that matches counts).  With NAVSLAM_RECORD_REF_DIGESTS set the answer is
    recorded instead of checked against the file."""
    mine = [digest(x) for x in (got, *also)]
    if ref_fn is not None:
        want = digest(ref_fn())
        assert want in mine, key
    else:
        want = mine[0]
    if _RECORD_TO:
        _recorded[key] = want
        return
    stored = stored_answers().get(key)
    if ref_fn is None:
        assert stored is not None, f"no stored reference answer for {key}"
        assert stored in mine, key
    elif stored is not None:
        assert stored == want, f"{key}: tests/golden/ref_digests.json differs from the reference"


def write_recorded(header: dict):
    """Write what check_ref() recorded, under `header`, to the file NAVSLAM_RECORD_REF_DIGESTS names."""
    with open(_RECORD_TO, "w") as f:
        json.dump({**header, "answers": dict(sorted(_recorded.items()))}, f, indent=0)
        f.write("\n")


class RefLib:
    """The reference's own compiled code for one MAX_ROWS x MAX_COLS shape."""

    def __init__(self, rows, cols):
        self.rows, self.cols = rows, cols
        path = os.path.join(REF_DIR, f"libnavref_{rows}x{cols}.so")
        self.lib = C.CDLL(path)
        L = self.lib
        assert L.refdrv_rows() == rows and L.refdrv_cols() == cols
        for f in ("refdrv_sizeof_pointcloud", "refdrv_sizeof_slam_attr", "refdrv_sizeof_kdnode",
                  "refdrv_sizeof_neighbor_result", "refdrv_offsetof_frame_count",
                  "refdrv_offsetof_trees", "refdrv_offsetof_error"):
            getattr(L, f).restype = C.c_size_t
        L.buildKDTree.restype = C.c_void_p
        L.buildKDTree.argtypes = [c_double_p, C.c_size_t, C.c_int]
        L.freeKDTree.argtypes = [C.c_void_p]
        L.nearestNeighborSearch.argtypes = [C.c_void_p, c_double_p, c_double_p, c_double_p, C.c_int]
        L.refdrv_nn_batch.restype = C.c_double
        L.refdrv_nn_batch.argtypes = [C.c_void_p, c_double_p, C.c_size_t, c_double_p, c_double_p]
        L.refdrv_build_rows.restype = C.c_double
        L.refdrv_build_rows.argtypes = [C.c_void_p, c_int_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
        L.refdrv_nn_rows.restype = C.c_double
        L.refdrv_nn_rows.argtypes = [C.POINTER(C.c_void_p), C.c_void_p, c_int_p, c_double_p, c_double_p,
                                     C.POINTER(C.c_size_t)]
        L.refdrv_free_rows.argtypes = [C.POINTER(C.c_void_p)]
        L.refdrv_extract_feature_timed.restype = C.c_double
        L.refdrv_extract_feature_timed.argtypes = [C.c_void_p, c_int_p, C.c_int]
        L.refdrv_build_timed.restype = C.c_double
        L.refdrv_build_timed.argtypes = [c_double_p, C.c_size_t, C.POINTER(C.c_void_p)]
        L.refdrv_tree_preorder.restype = C.c_size_t
        L.refdrv_tree_preorder.argtypes = [C.c_void_p, c_double_p, c_int_p, C.c_size_t]
        L.extract_feature.argtypes = [C.c_void_p, c_int_p]
        L.flattenPoints.argtypes = [c_double_p, c_int_p, c_double_p, C.POINTER(C.c_size_t)]
        L.convertToPointCloud.argtypes = [c_int_p, c_double_p]
        L.getRotationMatrix.argtypes = [C.c_double, C.c_double, C.c_double, c_double_p]
        L.init_slam.argtypes = [C.c_void_p, Pos, C.c_void_p]
        L.slam_mapping.argtypes = [C.c_void_p, Pos, C.c_void_p]
        L.slam_localization.restype = Pos
        L.slam_localization.argtypes = [C.c_void_p, C.c_void_p, Pos, Pos]
        L.refdrv_l9_read.restype = C.c_double
        L.refdrv_l9_read.argtypes = [C.c_char_p, C.c_void_p, C.POINTER(C.c_size_t)]
        self.sizeof_pointcloud = L.refdrv_sizeof_pointcloud()
        self.sizeof_slam_attr = L.refdrv_sizeof_slam_attr()

    def l5_json_read(self, path, max_frames, fill=0):
        """The reference's own LidarProcessData (jansson) into pre-filled L5_LidarDataFrame structs.
        Returns (distances [n,R,C] int32, timestamps [n] int32)."""
        L = self.lib
        L.refdrv_sizeof_l5_frame.restype = C.c_size_t
        L.refdrv_l5_json_read.restype = C.c_size_t
        L.refdrv_l5_json_read.argtypes = [C.c_char_p, C.c_void_p]
        sz = L.refdrv_sizeof_l5_frame()
        assert sz == 4 + 4 * self.rows * self.cols
        buf = np.full((max_frames, sz // 4), fill, dtype=np.int32)
        with quiet_stdout():
            n = L.refdrv_l5_json_read(path.encode(), buf.ctypes.data)
        return buf[:n, 1:].reshape(n, self.rows, self.cols).copy(), buf[:n, 0].copy()

    def imu_json_read(self, path, max_frames):
        """The reference's own IMUProcessData.  Returns (params [n,6] roll,pitch,yaw,x,y,z, timestamps [n])."""
        L = self.lib
        L.refdrv_sizeof_imu_frame.restype = C.c_size_t
        L.refdrv_imu_json_read.restype = C.c_size_t
        L.refdrv_imu_json_read.argtypes = [C.c_char_p, C.c_void_p]
        assert L.refdrv_sizeof_imu_frame() == 56
        buf = np.zeros((max_frames, 7), dtype=np.float64)
        with quiet_stdout():
            n = L.refdrv_imu_json_read(path.encode(), buf.ctypes.data)
        ts = buf[:n, 0].copy().view(np.int32)[::2].copy()
        return buf[:n, 1:].copy(), ts

    def l9_csv_read(self, path, max_frames):
        """The reference's own L9_LidarProcessData into zeroed PointCloud structs.
        Returns (frames [n,R,C,3], timestamps [n], seconds)."""
        buf = np.zeros((max_frames, self.sizeof_pointcloud), dtype=np.uint8)
        n = C.c_size_t(0)
        secs = self.lib.refdrv_l9_read(path.encode(), buf.ctypes.data, C.byref(n))
        ts = buf[:n.value, :4].copy().view(np.int32).reshape(-1)
        pts = buf[:n.value, 8:].copy().view(np.float64).reshape(n.value, self.rows, self.cols, 3)
        return pts, ts, secs

    # PointCloud = {int ts; Point pts[R][C]} with the points at byte offset 8
    def pack_cloud(self, cloud, ts=0) -> np.ndarray:
        cloud = _pts(cloud)
        buf = np.zeros(self.sizeof_pointcloud, dtype=np.uint8)
        buf[:4] = np.frombuffer(np.int32(ts).tobytes(), dtype=np.uint8)
        buf[8:] = np.frombuffer(cloud.tobytes(), dtype=np.uint8)
        return buf

    def extract_feature(self, cloud, feature=None):
        pc = self.pack_cloud(cloud)
        if feature is None:
            feature = np.zeros((self.rows, self.cols), dtype=np.int32)
        self.lib.extract_feature(pc.ctypes.data, _ip(feature))
        return feature

    def time_extract_feature(self, cloud, reps=5):
        pc = self.pack_cloud(cloud)
        feature = np.zeros((self.rows, self.cols), dtype=np.int32)
        return self.lib.refdrv_extract_feature_timed(pc.ctypes.data, _ip(feature), reps)

    def flatten(self, row, feat):
        row = _pts(row)
        feat = np.ascontiguousarray(feat, dtype=np.int32)
        out = np.empty_like(row)
        n = C.c_size_t(0)
        self.lib.flattenPoints(_dp(row), _ip(feat), _dp(out), C.byref(n))
        return out[:n.value].copy()

    def convert(self, dist):
        dist = np.ascontiguousarray(dist, dtype=np.int32)
        out = np.empty((self.rows, self.cols, 3))
        self.lib.convertToPointCloud(_ip(dist), _dp(out))
        return out

    def rotation(self, roll, pitch, yaw):
        R = np.empty(9)
        self.lib.getRotationMatrix(roll, pitch, yaw, _dp(R))
        return R

    def tree_build(self, pts, timed=False):
        work = _pts(pts).copy()
        if timed:
            root = C.c_void_p()
            dt = self.lib.refdrv_build_timed(_dp(work), work.shape[0], C.byref(root))
            return root.value, work, dt
        return self.lib.buildKDTree(_dp(work), work.shape[0], 0), work

    def tree_free(self, h):
        self.lib.freeKDTree(h)

    def tree_preorder(self, h, n):
        out = np.empty((n, 3))
        depth = np.empty(n, dtype=np.int32)
        k = self.lib.refdrv_tree_preorder(h, _dp(out), _ip(depth), n)
        return out[:k], depth[:k]

    def nn_batch(self, h, q):
        q = _pts(q)
        out = np.full_like(q, np.nan)
        dist = np.empty(q.shape[0])
        dt = self.lib.refdrv_nn_batch(h, _dp(q), q.shape[0], _dp(out), _dp(dist))
        return out, dist, dt

    def build_rows(self, global_cloud, feature):
        pc = self.pack_cloud(global_cloud)
        feature = np.ascontiguousarray(feature, dtype=np.int32)
        trees = (C.c_void_p * self.rows)()
        counts = (C.c_size_t * self.rows)()
        dt = self.lib.refdrv_build_rows(pc.ctypes.data, _ip(feature), trees, counts)
        return trees, np.array(list(counts)), dt

    def nn_rows(self, trees, queries, feature):
        pc = self.pack_cloud(queries)
        feature = np.ascontiguousarray(feature, dtype=np.int32)
        out = np.full((self.rows, self.cols, 3), np.nan)
        dist = np.empty((self.rows, self.cols))
        nq = C.c_size_t(0)
        dt = self.lib.refdrv_nn_rows(trees, pc.ctypes.data, _ip(feature), _dp(out), _dp(dist), C.byref(nq))
        return out, dist, nq.value, dt

    def free_rows(self, trees):
        self.lib.refdrv_free_rows(trees)

    # whole step on a heap-allocated SLAM_attr (315 MB at 64x2048, SURVEY D6)
    def new_attr(self) -> np.ndarray:
        return np.zeros(self.sizeof_slam_attr, dtype=np.uint8)

    def attr_global(self, attr, frame) -> np.ndarray:
        off = frame * self.sizeof_pointcloud + 8
        n = self.rows * self.cols * 24
        return np.frombuffer(attr[off:off + n].tobytes(), dtype=np.float64).reshape(self.rows, self.cols, 3)

    def attr_frame_count(self, attr) -> int:
        off = self.lib.refdrv_offsetof_frame_count()
        return int(np.frombuffer(attr[off:off + 4].tobytes(), dtype=np.int32)[0])

    def attr_set_frame_count(self, attr, v):
        off = self.lib.refdrv_offsetof_frame_count()
        attr[off:off + 4] = np.frombuffer(np.int32(v).tobytes(), dtype=np.uint8)

    def attr_error(self, attr) -> float:
        off = self.lib.refdrv_offsetof_error()
        return float(np.frombuffer(attr[off:off + 8].tobytes(), dtype=np.float64)[0])

    def init_slam(self, attr, pos, cloud):
        pc = self.pack_cloud(cloud)
        self.lib.init_slam(attr.ctypes.data, Pos.of(pos), pc.ctypes.data)

    def slam_mapping(self, attr, pos, cloud):
        pc = self.pack_cloud(cloud)
        self.lib.slam_mapping(attr.ctypes.data, Pos.of(pos), pc.ctypes.data)

    def slam_localization(self, attr, cloud, pos_predict, pos_last):
        pc = self.pack_cloud(cloud)
        with quiet_stdout():
            out = self.lib.slam_localization(attr.ctypes.data, pc.ctypes.data, Pos.of(pos_predict),
                                             Pos.of(pos_last))
        return out.arr()
