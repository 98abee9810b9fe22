"""CPU-only checks of the drop-in boundary: the C-ABI library loads and exports every symbol
include/navslam_b200.h declares, the per-shape shims export the reference's symbols with the
reference's struct layouts, and the product fails loudly without a GPU (no CPU fallback)."""
import ctypes as C
import importlib
import os
import re

import numpy as np
import pytest

from oracle_lib import RefLib, check_ref, ref_available

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [(8, 8), (5, 33), (16, 1800), (64, 2048)]
REF_SYMBOLS = ["convertToPointCloud", "printPointCloud", "init_slam", "slam_localization", "slam_mapping",
               "printKDTree", "buildKDTree", "freeKDTree", "nearestNeighborSearch", "extract_feature",
               "flattenPoints", "compute_posdiff", "getRotationMatrix", "getAxis", "euclideanDistance",
               "mapCoordinatesToLastFrame", "nth_element"]


@pytest.fixture(scope="module")
def built(pkg):
    pkg.build.build_all()
    return pkg


def test_library_exports_every_declared_symbol(built):
    hdr = open(os.path.join(ROOT, "include", "navslam_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(nav_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 35
    L = C.CDLL(built.build.LIB)
    missing = [s for s in declared if not hasattr(L, s)]
    assert not missing, missing
    binding = importlib.import_module("nav-slam_b200.binding")
    assert sorted(binding.EXPORTS) == declared


@pytest.mark.parametrize("shape", SHAPES)
def test_shim_exports_reference_symbols_and_layouts(built, shape):
    so = built.build.shim_path(*shape)
    assert os.path.exists(so)
    S = C.CDLL(so)
    for sym in REF_SYMBOLS:
        assert hasattr(S, sym), sym
    for f in ("sizeof_pointcloud", "sizeof_slam_attr", "sizeof_kdnode", "sizeof_neighbor_result",
              "offsetof_frame_count", "offsetof_trees", "offsetof_error"):
        getattr(S, "navslam_abi_" + f).restype = C.c_size_t
    r, c = shape
    assert (S.navslam_abi_rows(), S.navslam_abi_cols()) == shape
    assert S.navslam_abi_sizeof_pointcloud() == 8 + r * c * 24
    assert S.navslam_abi_sizeof_slam_attr() == 100 * (8 + r * c * 24) + 8 + r * 8 + 8
    names = ("sizeof_pointcloud", "sizeof_slam_attr", "sizeof_kdnode", "sizeof_neighbor_result",
             "offsetof_frame_count", "offsetof_trees", "offsetof_error")
    ref = RefLib(r, c).lib if ref_available(f"{r}x{c}") else None
    check_ref(f"abi_layout/{r}x{c}", np.array([getattr(S, "navslam_abi_" + f)() for f in names], dtype=np.int64),
              ref and (lambda: np.array([getattr(ref, "refdrv_" + f)() for f in names], dtype=np.int64)))


def test_fails_loudly_without_a_gpu(built):
    if built.device_count() > 0:
        pytest.skip("a CUDA device is visible here")
    with pytest.raises(built.NavError, match="no CUDA device"):
        built.Context(8, 8)
    with pytest.raises(built.NavError, match="no CUDA device"):
        built.KdTree([[0.0, 0.0, 0.0]])


def test_product_never_imports_the_oracle():
    """nothing under nav-slam_b200/ may reference oracle/ (the checker is test infrastructure)"""
    bad = []
    pk = os.path.join(ROOT, "nav-slam_b200")
    for dirpath, _, files in os.walk(pk):
        if "_build" in dirpath or "__pycache__" in dirpath:
            continue
        for fn in files:
            if not fn.endswith((".py", ".cu", ".cuh", ".c", ".h")):
                continue
            txt = open(os.path.join(dirpath, fn), errors="replace").read()
            if re.search(r"navslam_oracle|oracle_lib|libnavoracle|libnavref|import oracle|from oracle", txt):
                bad.append(os.path.join(dirpath, fn))
            if fn == "build.py":
                continue
    # build.py may *link* the reference's main.o against the shim (a test artefact kept in oracle/_ref)
    bad = [b for b in bad if not b.endswith("build.py")]
    assert not bad, bad


def test_shim_host_helpers_match_reference(built):
    """nth_element and mapCoordinatesToLastFrame are plain host code in the shim: same results as the
    reference's compiled functions (oracle/_ref where built, else their stored answers), no GPU involved."""
    S = C.CDLL(built.build.shim_path(8, 8))
    R = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libnavref_8x8.so")) if ref_available("8x8") else None
    libs = (S,) if R is None else (S, R)
    for L in libs:
        L.nth_element.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int]
        L.nth_element.restype = None
        L.mapCoordinatesToLastFrame.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.mapCoordinatesToLastFrame.restype = None
    rng = np.random.default_rng(3)
    for n in (1, 2, 7, 64, 501):
        for axis in (0, 1, 2):
            pts = np.round(rng.normal(0, 50, (n, 3)))          # rounded: plenty of equal keys
            a, b = pts.copy(), pts.copy()
            S.nth_element(a.ctypes.data, 0, n - 1, n // 2, axis)
            if R is not None:
                R.nth_element(b.ctypes.data, 0, n - 1, n // 2, axis)
            check_ref(f"nth_element/{n}/{axis}", a, R and (lambda: b))
    cloud = np.zeros(8 + 8 * 8 * 24, dtype=np.uint8)
    pts = rng.normal(0, 1000, (8, 8, 3))
    cloud[8:] = np.frombuffer(pts.tobytes(), dtype=np.uint8)
    tr = np.array([12.5, -3.25, 100.0])
    outs = []
    for L in libs:
        out = np.zeros_like(cloud)
        L.mapCoordinatesToLastFrame(cloud.ctypes.data, tr.ctypes.data, out.ctypes.data)
        outs.append(out[8:].copy().view(np.float64))
    check_ref("mapCoordinatesToLastFrame", outs[0], R and (lambda: outs[1]))
    assert np.array_equal(outs[0].reshape(8, 8, 3), pts - tr)
