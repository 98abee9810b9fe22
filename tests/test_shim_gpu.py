"""GPU tests of the drop-in shim: the reference's own symbols (init_slam, slam_localization,
slam_mapping, ...) served by libnavslam_shim_<RxC>.so, and the reference's UNMODIFIED main.c +
ekf.c linked against it (oracle/_ref/navshim_main_*), compared with the reference itself.  The two
whole-program tests need the reference's sources at build time and skip without them."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import big_stack
from oracle_lib import Pos, REF_DIR, RefLib, check_ref, quiet_stdout, ref_available

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class Shim:
    def __init__(self, pkg, rows, cols):
        self.rows, self.cols = rows, cols
        self.lib = C.CDLL(pkg.build.shim_path(rows, cols))
        L = self.lib
        L.navslam_abi_sizeof_slam_attr.restype = C.c_size_t
        L.navslam_abi_offsetof_frame_count.restype = C.c_size_t
        L.navslam_abi_offsetof_error.restype = C.c_size_t
        L.init_slam.argtypes = [C.c_void_p, Pos, C.c_void_p]
        L.slam_mapping.argtypes = [C.c_void_p, Pos, C.c_void_p]
        L.slam_localization.restype = Pos
        L.slam_localization.argtypes = [C.c_void_p, C.c_void_p, Pos, Pos]
        L.extract_feature.argtypes = [C.c_void_p, C.c_void_p]
        L.buildKDTree.restype = C.c_void_p
        L.buildKDTree.argtypes = [C.c_void_p, C.c_size_t, C.c_int]
        L.freeKDTree.argtypes = [C.c_void_p]
        L.nearestNeighborSearch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        self.pc_bytes = 8 + rows * cols * 24
        self.attr = np.zeros(L.navslam_abi_sizeof_slam_attr(), dtype=np.uint8)

    def pack(self, cloud, ts=0):
        buf = np.zeros(self.pc_bytes, dtype=np.uint8)
        buf[:4] = np.frombuffer(np.int32(ts).tobytes(), dtype=np.uint8)
        buf[8:] = np.frombuffer(np.ascontiguousarray(cloud, dtype=np.float64).tobytes(), dtype=np.uint8)
        return buf

    def global_cloud(self, frame):
        off = frame * self.pc_bytes + 8
        n = self.rows * self.cols * 24
        return np.frombuffer(self.attr[off:off + n].tobytes(), dtype=np.float64).reshape(self.rows, self.cols, 3)

    def error(self):
        off = self.lib.navslam_abi_offsetof_error()
        return float(np.frombuffer(self.attr[off:off + 8].tobytes(), dtype=np.float64)[0])

    def frame_count(self):
        off = self.lib.navslam_abi_offsetof_frame_count()
        return int(np.frombuffer(self.attr[off:off + 4].tobytes(), dtype=np.int32)[0])


SLAM_STEP_CASES = [((8, 8), 8), ((5, 33), 6), ((64, 2048), 3)]


def reference_slam_steps(oracle, synth, shape, frames):
    """The reference's init_slam / slam_localization / slam_mapping on the shim test's inputs: the oracle in
    the reference's tie mode, checked against the reference (live where oracle/_ref is built, else its stored
    answers).  Returns the clouds, the start pose and per frame (pose, error, global cloud)."""
    r, c = shape
    key = f"shim_slam_step/{r}x{c}"
    ref = RefLib(r, c) if ref_available(f"{r}x{c}") else None
    if shape == (8, 8):
        clouds = [oracle.convert(synth.l5_depth_frame(f)) for f in range(frames)]
    else:
        clouds = [synth.room_frame(r, c, f) for f in range(frames)]
    attr = ref.new_attr() if ref is not None else None
    slam = oracle.slam(r, c, 0)
    pos = np.array([10.0, -20.0, 5.0, 1.0, -2.0, 30.0])
    if ref is not None:
        big_stack(ref.init_slam, attr, pos, clouds[0])
    g = slam.init(pos, clouds[0])
    check_ref(f"{key}/global0", g, ref and (lambda: ref.attr_global(attr, 0)))
    steps = [(pos, 0.0, g)]
    last = pos
    for f in range(1, frames):
        pred = last + np.array([45.0, 3.0, -1.0, 0.0, 0.0, 0.0])
        p, _, err, _ = slam.localize(clouds[f], pred, last)
        if ref is not None:
            p_ref = big_stack(ref.slam_localization, attr, clouds[f], pred, last)
            big_stack(ref.slam_mapping, attr, p_ref, clouds[f])
            assert ref.attr_frame_count(attr) == f + 1
        check_ref(f"{key}/pose{f}", p, ref and (lambda: p_ref))
        check_ref(f"{key}/error{f}", np.float64(err), ref and (lambda: np.float64(ref.attr_error(attr))))
        g = slam.map(p, clouds[f])
        check_ref(f"{key}/global{f}", g, ref and (lambda: ref.attr_global(attr, f)))
        steps.append((p, err, g))
        last = p
    slam.close()
    return clouds, pos, steps


@pytest.mark.parametrize("shape,frames", SLAM_STEP_CASES)
def test_shim_slam_step_matches_reference(pkg, oracle, synth, shape, frames):
    r, c = shape
    clouds, pos, steps = reference_slam_steps(oracle, synth, shape, frames)
    shim = Shim(pkg, r, c)
    pc = shim.pack(clouds[0], 7)
    shim.lib.init_slam(shim.attr.ctypes.data, Pos.of(pos), pc.ctypes.data)
    assert np.array_equal(shim.global_cloud(0), steps[0][2])
    assert shim.frame_count() == 1
    last = pos
    for f in range(1, frames):
        p_ref, err_ref, g_ref = steps[f]
        pred = last + np.array([45.0, 3.0, -1.0, 0.0, 0.0, 0.0])
        pc = shim.pack(clouds[f], 7 + f)
        with quiet_stdout():
            p = shim.lib.slam_localization(shim.attr.ctypes.data, pc.ctypes.data, Pos.of(pred), Pos.of(last)).arr()
        assert np.array_equal(p, p_ref), (f, p - p_ref)
        assert shim.error() == err_ref
        shim.lib.slam_mapping(shim.attr.ctypes.data, Pos.of(p), pc.ctypes.data)
        assert np.array_equal(shim.global_cloud(f), g_ref)
        assert shim.frame_count() == f + 1
        last = p_ref


def test_shim_function_level_symbols(pkg, oracle, synth):
    shape = (5, 33)
    shim = Shim(pkg, *shape)
    cloud = synth.room_frame(*shape, 1)
    feat = np.zeros(shape, dtype=np.int32)
    pc = shim.pack(cloud)  # keep the buffer alive across the call
    shim.lib.extract_feature(pc.ctypes.data, feat.ctypes.data)
    assert np.array_equal(feat, oracle.extract_feature(cloud))
    pts = synth.map_points(5000, seed=9)
    q = synth.map_queries(pts, 20, seed=10)
    work = pts.copy()
    h = shim.lib.buildKDTree(work.ctypes.data, work.shape[0], 0)
    oi, od = oracle.nn_brute(pts, q)
    for i in range(q.shape[0]):
        best = np.array([np.inf])
        out = np.full(3, np.nan)
        tq = q[i].copy()
        shim.lib.nearestNeighborSearch(h, tq.ctypes.data, out.ctypes.data, best.ctypes.data, 0)
        assert best[0] == od[i] and np.array_equal(out, pts[oi[i]])
        # a caller-supplied bound below the true distance leaves the outputs untouched (kdtree.c:117)
        best = np.array([od[i] * 0.5])
        out = np.full(3, np.nan)
        shim.lib.nearestNeighborSearch(h, tq.ctypes.data, out.ctypes.data, best.ctypes.data, 0)
        assert best[0] == od[i] * 0.5 and np.isnan(out).all()
    shim.lib.freeKDTree(h)
    assert shim.lib.buildKDTree(work.ctypes.data, 0, 0) is None


def _run_main(exe, workdir, files, args=()):
    os.makedirs(workdir, exist_ok=True)
    for name, text in files.items():
        with open(os.path.join(workdir, name), "w") as f:
            f.write(text)
    res = subprocess.run([exe, *args], cwd=workdir, capture_output=True, timeout=600)
    assert res.returncode == 0, res.stderr.decode(errors="replace")[-2000:]
    with open(os.path.join(workdir, "point_cloud_data.csv"), "rb") as f:
        return res.stdout, f.read()


def test_unmodified_main_l5_config1(synth, tmp_path):
    """BASELINE config 1: the reference's main.c L5 handler on a synthetic parsed_data.json, once as
    the reference program and once linked against the B200 shim: identical stdout and CSV."""
    ref_exe = os.path.join(REF_DIR, "navref_main_8x8")
    shim_exe = os.path.join(REF_DIR, "navshim_main_8x8")
    if not (os.path.exists(ref_exe) and os.path.exists(shim_exe)):
        pytest.skip("reference mains not built (needs /root/reference at build time)")
    js = synth.l5_json(30)
    out_ref, csv_ref = _run_main(ref_exe, str(tmp_path / "ref"), {"parsed_data.json": js})
    out_shim, csv_shim = _run_main(shim_exe, str(tmp_path / "shim"), {"parsed_data.json": js})
    assert csv_ref.count(b"\n") == 1 + 30 * 64
    assert csv_shim == csv_ref
    assert out_shim == out_ref


def test_unmodified_main_l9_config2(synth, tmp_path):
    """BASELINE config 2: L9 handler, 16x1800 integer-mm CSV.  Integer data has exact distance ties,
    where the shim picks the lowest index and the reference the first DFS visit, so the fitted poses
    may differ far below the CSV's %.2f resolution; the CSVs are compared numerically."""
    ref_exe = os.path.join(REF_DIR, "navref_l9_16x1800")
    shim_exe = os.path.join(REF_DIR, "navshim_l9_16x1800")
    if not (os.path.exists(ref_exe) and os.path.exists(shim_exe)):
        pytest.skip("reference mains not built (needs /root/reference at build time)")
    csv_in = synth.l9_csv(synth.l9_sequence(4))
    _, csv_ref = _run_main(ref_exe, str(tmp_path / "ref"), {"parsed_data.csv": csv_in})
    _, csv_shim = _run_main(shim_exe, str(tmp_path / "shim"), {"parsed_data.csv": csv_in})
    a = np.genfromtxt(csv_ref.decode().splitlines(), delimiter=",", skip_header=1)
    b = np.genfromtxt(csv_shim.decode().splitlines(), delimiter=",", skip_header=1)
    assert a.shape == b.shape == (4 * 16 * 1800, 25)
    assert np.abs(a - b).max() <= 0.011
    same = (csv_ref == csv_shim)
    print("L9 CSV byte-identical:", same)


@pytest.mark.gpu
def test_shim_fast_modes_agree(synth, tmp_path):
    """NAVSLAM_ADAM=stats with and without NAVSLAM_TRUST_FRAME / NAVSLAM_PIN (the shim page-locks the caller's
    PointCloud and SLAM_attr where they lie): identical poses and identical mapped clouds.  The modes are read
    once per process, so every combination runs in a process of its own."""
    import json
    import subprocess
    import sys
    code = r'''
import importlib, json, sys, os
import numpy as np
sys.path.insert(0, %r)
nav = importlib.import_module("nav-slam_b200")
sb = importlib.import_module("nav-slam_b200.shim_binding")
R, C_ = 16, 1800
frames = nav.synth.room_sequence(R, C_, 4, cfg=2, elev=(-15.0, 15.0))
shim = sb.ShimSlam(R, C_)
pc = shim.pack_cloud(frames[0], ts=0)
fd = os.dup(1); os.dup2(os.open(os.devnull, os.O_WRONLY), 1)
shim.init_slam(np.zeros(6), pc)
last = np.zeros(6); poses = []
for f in range(1, 4):
    pc[8:] = frames[f].reshape(-1).view(np.uint8)
    p = shim.slam_localization(pc, last + np.array([48.0, 0.5, 0, 0, 0, 0]), last)
    shim.slam_mapping(p, pc)
    poses.append([float(v).hex() for v in p]); last = p
g = shim.global_cloud(3).copy()
os.dup2(fd, 1)
print(json.dumps({"poses": poses, "sum": float(g.sum()).hex(), "fc": shim.frame_count}))
shim.release()
''' % ROOT
    outs = {}
    for name, env in (("stats", {"NAVSLAM_ADAM": "stats"}),
                      ("trust", {"NAVSLAM_ADAM": "stats", "NAVSLAM_TRUST_FRAME": "1"}),
                      ("pinned", {"NAVSLAM_ADAM": "stats", "NAVSLAM_TRUST_FRAME": "1", "NAVSLAM_PIN": "1"})):
        e = {k: v for k, v in os.environ.items() if not k.startswith("NAVSLAM_")}
        e.update(env)
        res = subprocess.run([sys.executable, "-c", code], env=e, capture_output=True, text=True, timeout=300)
        assert res.returncode == 0, res.stderr[-2000:]
        outs[name] = json.loads(res.stdout.strip().splitlines()[-1])
    assert outs["stats"] == outs["trust"] == outs["pinned"]
    assert outs["stats"]["fc"] == 4   # init_slam + three mapped frames
