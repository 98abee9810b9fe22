"""Pins the oracle: every function of oracle/navslam_oracle.c must be bit-identical to the
reference's own code on seeded inputs: live against oracle/_ref/libnavref_<RxC>.so where
oracle/build_ref.sh built it from the reference's sources, otherwise against the reference's
answers stored as digests in tests/golden/ref_digests.json (oracle_lib.check_ref).  CPU only."""
import ctypes as C

import numpy as np
import pytest

from conftest import big_stack
from oracle_lib import RefLib, check_ref, ref_available

SHAPES = [(8, 8), (5, 33), (16, 1800), (64, 2048)]


def _ref(shape):
    """RefLib where oracle/_ref is built, else None (check_ref then uses the stored answers)."""
    return RefLib(*shape) if ref_available(f"{shape[0]}x{shape[1]}") else None


def _live(ref, fn):
    return None if ref is None else fn


def _cloud(synth, shape, frame=0, **kw):
    r, c = shape
    if shape == (16, 1800):
        return synth.room_frame(r, c, frame, cfg=2, elev=(-15, 15), integer_mm=True, **kw)
    return synth.room_frame(r, c, frame, **kw)


def _name(shape):
    return f"{shape[0]}x{shape[1]}"


@pytest.mark.parametrize("shape", SHAPES)
def test_struct_sizes(pkg, shape):
    """The reference's struct sizes, as the product's shim lays them out for the same shape."""
    ref = _ref(shape)
    r, c = shape
    shim = C.CDLL(pkg.build.shim_path(r, c))
    names = ("sizeof_pointcloud", "sizeof_slam_attr", "sizeof_kdnode", "sizeof_neighbor_result")
    for f in names:
        getattr(shim, "navslam_abi_" + f).restype = C.c_size_t
    sizes = np.array([getattr(shim, "navslam_abi_" + f)() for f in names], dtype=np.int64)
    assert sizes.tolist() == [8 + r * c * 24, 100 * (8 + r * c * 24) + 8 + r * 8 + 8, 40, 56]
    check_ref(f"struct_sizes/{_name(shape)}", sizes, _live(ref, lambda: np.array(
        [ref.sizeof_pointcloud, ref.sizeof_slam_attr, ref.lib.refdrv_sizeof_kdnode(),
         ref.lib.refdrv_sizeof_neighbor_result()], dtype=np.int64)))


@pytest.mark.parametrize("shape", SHAPES)
def test_extract_feature_bit_exact(oracle, synth, shape):
    ref = _ref(shape)
    for frame, inv in ((0, 0.0), (3, 0.02)):
        cloud = _cloud(synth, shape, frame, invalid_frac=inv)
        b = oracle.extract_feature(cloud)
        check_ref(f"extract_feature/{_name(shape)}/{frame}", b, _live(ref, lambda: ref.extract_feature(cloud)))
        assert b[:, :2].sum() == 0 and b[:, -2:].sum() == 0
        curv = oracle.curvature(cloud)
        assert np.array_equal(curv > 0.1, b == 1)
    # never writes zeros: pre-set labels survive
    pre = np.full(shape, 7, dtype=np.int32)
    b = oracle.extract_feature(cloud, pre.copy())
    check_ref(f"extract_feature/{_name(shape)}/preset", b, _live(ref, lambda: ref.extract_feature(cloud, pre.copy())))
    assert set(np.unique(b)) <= {1, 7}


def test_extract_feature_special_values(oracle):
    ref = _ref((5, 33))
    rng = np.random.default_rng(7)
    cloud = rng.normal(0, 1000, size=(5, 33, 3))
    cloud[0, 5] = np.nan
    cloud[1, 7] = np.inf
    cloud[2, 10:20] = 0.0          # run of invalid returns
    cloud[3, :] = cloud[3, 0]      # all equal -> avg 0
    cloud[4, 10:14] = 1e-200       # underflowing squares
    check_ref("extract_feature/special_values", oracle.extract_feature(cloud),
              _live(ref, lambda: ref.extract_feature(cloud)))


def test_collinear_equal_spacing_is_edge(oracle):
    # SURVEY D10: equally spaced collinear neighbours give 0.25/2.25 = 1/9 > 0.1
    cloud = np.zeros((1, 16, 3))
    cloud[0, :, 0] = 100.0 * np.arange(16)
    curv = oracle.curvature(cloud)
    assert np.allclose(curv[0, 2:-2], 1.0 / 9.0, rtol=1e-6)
    assert oracle.extract_feature(cloud)[0, 2:-2].all()


@pytest.mark.parametrize("shape", [(8, 8), (5, 33)])
def test_convert_bit_exact(oracle, synth, shape):
    ref = _ref(shape)
    rng = np.random.default_rng(11)
    d = rng.integers(-5, 4000, size=shape).astype(np.int32)
    d[0, 0] = 0
    check_ref(f"convert/{_name(shape)}/random", oracle.convert(d), _live(ref, lambda: ref.convert(d)))
    d8 = synth.l5_depth_frame(3, *shape)
    check_ref(f"convert/{_name(shape)}/l5", oracle.convert(d8), _live(ref, lambda: ref.convert(d8)))


def test_rotation_and_transform_bit_exact(oracle, synth):
    ref = _ref((5, 33))
    rng = np.random.default_rng(5)
    poses = [np.concatenate([rng.normal(0, 5000, 3), rng.uniform(-180, 180, 3)]) for _ in range(20)]
    got = np.stack([oracle.rotation_deg(pos) for pos in poses])
    check_ref("rotation/20_poses", got, _live(ref, lambda: np.stack(
        [ref.rotation(pos[3] * np.pi / 180.0, pos[4] * np.pi / 180.0, pos[5] * np.pi / 180.0) for pos in poses])))


@pytest.mark.parametrize("shape", SHAPES)
def test_flatten_bit_exact(oracle, synth, shape):
    ref = _ref(shape)
    cloud = _cloud(synth, shape, 1)
    feat = oracle.extract_feature(cloud)
    feat[0, 0] = 1
    feat[-1, -1] = 1
    feat[0, 1] = 2  # only ==1 is selected (src/slam.c:68)
    for r in (0, shape[0] - 1):
        check_ref(f"flatten/{_name(shape)}/row{r}", oracle.flatten(cloud[r], feat[r]),
                  _live(ref, lambda: ref.flatten(cloud[r], feat[r])))


@pytest.mark.parametrize("kind", ["uniform", "clustered", "integer", "duplicates", "sorted"])
@pytest.mark.parametrize("n", [0, 1, 2, 3, 17, 1000, 20000])
def test_tree_build_and_nn_bit_exact(oracle, synth, kind, n):
    ref = _ref((8, 8))
    key = f"tree/{kind}/{n}"
    rng = np.random.default_rng(n + 13)
    if kind == "uniform":
        pts = synth.map_points(n, seed=n)
    elif kind == "clustered":
        pts = synth.map_points(n, variant="clustered", seed=n)
    elif kind == "integer":
        pts = rng.integers(0, 50, size=(n, 3)).astype(np.float64)  # many equal keys + exact ties
    elif kind == "duplicates":
        pts = np.repeat(rng.normal(0, 100, size=((n + 3) // 4, 3)), 4, axis=0)[:n]
    else:
        pts = np.stack([np.arange(n, dtype=np.float64)] * 3, axis=1)  # Lomuto worst case (quadratic select)
    h_ref, perm_ref = ref.tree_build(pts) if ref is not None else (None, None)
    h_or, perm_or = oracle.tree_build(pts)
    check_ref(key + "/perm", perm_or, _live(ref, lambda: perm_ref))   # same in-place permutation
    if n:
        b, db = oracle.tree_preorder(h_or, n)
        a, da = ref.tree_preorder(h_ref, n) if ref is not None else (None, None)
        check_ref(key + "/preorder", b, _live(ref, lambda: a))
        check_ref(key + "/depth", db, _live(ref, lambda: da))
    nq = 300
    q = (pts[rng.integers(0, n, size=nq)] + rng.normal(0, 3, size=(nq, 3))) if n else rng.normal(size=(nq, 3))
    if kind == "integer":
        q = np.rint(q)
    p_or, d_or = oracle.tree_nn(h_or, q)
    p_ref, d_ref, _ = ref.nn_batch(h_ref, q) if ref is not None else (None, None, None)
    check_ref(key + "/nn_dist", d_or, _live(ref, lambda: d_ref))
    check_ref(key + "/nn_point", p_or, _live(ref, lambda: p_ref))
    # from here on p_or / d_or stand for the reference's answers (equal, checked above)
    # canonical form: same distance always; same point unless an exact distance tie exists
    idx, d_can = oracle.nn_brute(pts, q)
    if n:
        assert np.array_equal(d_can, d_or)
        ties = oracle.nn_tie_count(pts, q)
        same = np.all(pts[idx] == p_or, axis=1)
        assert np.all(same | (ties > 1))
        # the reference's answer is always one of the tied candidates
        d_back = np.sqrt(((p_or - q) ** 2)[:, 0] + ((p_or - q) ** 2)[:, 1] + ((p_or - q) ** 2)[:, 2])
        assert np.array_equal(d_back, d_or)
    else:
        assert np.all(idx == -1) and np.all(np.isinf(d_can)) and np.all(np.isinf(d_or))
    if ref is not None:
        ref.tree_free(h_ref)
    oracle.tree_free(h_or)


@pytest.mark.parametrize("shape", [(8, 8), (5, 33), (16, 1800)])
def test_whole_step_bit_exact(oracle, synth, shape):
    """init_slam / slam_localization / slam_mapping (reference tie mode) vs the reference."""
    ref = _ref(shape)
    r, c = shape
    key = f"whole_step/{_name(shape)}"
    frames = 6 if shape != (16, 1800) else 3
    attr = ref.new_attr() if ref is not None else None
    slam = oracle.slam(r, c, 0)
    if shape == (8, 8):
        clouds = [oracle.convert(synth.l5_depth_frame(f)) for f in range(frames)]
    else:
        clouds = [_cloud(synth, shape, f) for f in range(frames)]
    pos = np.array([10.0, -20.0, 5.0, 1.0, -2.0, 30.0])
    if ref is not None:
        big_stack(ref.init_slam, attr, pos, clouds[0])
    g = slam.init(pos, clouds[0])
    check_ref(f"{key}/global0", g, _live(ref, lambda: ref.attr_global(attr, 0)))
    last = pos
    for f in range(1, frames):
        pred = last + np.array([45.0, 3.0, -1.0, 0.0, 0.0, 0.0])
        p_or, corr, err, iters = slam.localize(clouds[f], pred, last)
        if ref is not None:
            p_ref = big_stack(ref.slam_localization, attr, clouds[f], pred, last)
        check_ref(f"{key}/pose{f}", p_or, _live(ref, lambda: p_ref))
        check_ref(f"{key}/error{f}", np.float64(err), _live(ref, lambda: np.float64(ref.attr_error(attr))))
        if ref is not None:
            big_stack(ref.slam_mapping, attr, p_ref, clouds[f])
        g = slam.map(p_or, clouds[f])
        check_ref(f"{key}/global{f}", g, _live(ref, lambda: ref.attr_global(attr, f)))
        if ref is not None:
            assert ref.attr_frame_count(attr) == f + 1
        last = p_or
    slam.close()
