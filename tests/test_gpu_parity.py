"""GPU parity tests: the CUDA path, called through the C ABI (include/navslam_b200.h), against the
CPU oracle on the same seeded inputs.  Integer / index outputs and all binary64 values are
compared bit-for-bit (np.array_equal), which is tighter than north_star's 1e-5 tolerance for
curvature and distances."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SHAPES = [(8, 8), (5, 33), (16, 1800), (64, 2048)]


def _cloud(synth, shape, frame=0, **kw):
    r, c = shape
    if shape == (16, 1800):
        return synth.room_frame(r, c, frame, cfg=2, elev=(-15, 15), integer_mm=True, **kw)
    return synth.room_frame(r, c, frame, **kw)


@pytest.fixture(scope="module")
def ctxs(pkg):
    made = {}

    def get(shape, n_seq=1):
        key = (shape, n_seq)
        if key not in made:
            made[key] = pkg.Context(shape[0], shape[1], device=0, n_seq=n_seq)
        return made[key]

    yield get
    for c in made.values():
        c.close()


# ------------------------------------------------------------------ a3 -----------------------
@pytest.mark.parametrize("shape", SHAPES + [(3, 4), (2, 5), (7, 300)])
def test_labels_and_curvature_bit_exact(ctxs, oracle, synth, shape):
    ctx = ctxs(shape)
    for frame, inv in ((0, 0.0), (5, 0.03)):
        cloud = _cloud(synth, shape, frame, invalid_frac=inv)
        assert np.array_equal(ctx.extract_feature(cloud), oracle.extract_feature(cloud))
        assert np.array_equal(ctx.curvature(cloud), oracle.curvature(cloud))


def test_labels_only_sets_ones(ctxs, oracle, synth):
    shape = (5, 33)
    cloud = _cloud(synth, shape, 2)
    pre = np.full(shape, 7, dtype=np.int32)
    got = ctxs(shape).extract_feature(cloud, pre.copy())
    want = oracle.extract_feature(cloud, pre.copy())
    assert np.array_equal(got, want) and set(np.unique(got)) <= {1, 7}


def test_labels_special_values(ctxs, oracle):
    rng = np.random.default_rng(7)
    cloud = rng.normal(0, 1000, size=(5, 33, 3))
    cloud[0, 5] = np.nan
    cloud[1, 7] = np.inf
    cloud[2, 10:20] = 0.0
    cloud[3, :] = cloud[3, 0]
    cloud[4, 10:14] = 1e-200
    cloud[4, 20:24] = 1e200
    ctx = ctxs((5, 33))
    assert np.array_equal(ctx.extract_feature(cloud), oracle.extract_feature(cloud))
    assert np.array_equal(ctx.curvature(cloud), oracle.curvature(cloud), equal_nan=True)


def test_labels_near_threshold(ctxs, oracle):
    """Points engineered to sit within ~1e-12 of the 0.1 threshold on both sides."""
    rng = np.random.default_rng(3)
    rows, cols = 5, 33
    cloud = np.zeros((rows, cols, 3))
    # collinear with spacing pattern s, s, t, t around each point: tune t so curvature ~ 0.1
    for r in range(rows):
        x = np.cumsum(rng.uniform(90, 110, size=cols))
        cloud[r, :, 0] = x
        cloud[r, :, 1] = rng.normal(0, 2.0, size=cols)
    ctx = ctxs((rows, cols))
    base = oracle.curvature(cloud)
    # bisect one coordinate of the centre point so its curvature straddles 0.1
    r, c = 2, 16
    lo, hi = -200.0, 200.0
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        cloud[r, c, 1] = mid
        v = oracle.curvature(cloud)[r, c]
        if v > 0.1:
            hi = mid
        else:
            lo = mid
    for y in (lo, hi, np.nextafter(lo, -np.inf), np.nextafter(hi, np.inf)):
        cloud[r, c, 1] = y
        assert np.array_equal(ctx.extract_feature(cloud), oracle.extract_feature(cloud))
        assert np.array_equal(ctx.curvature(cloud), oracle.curvature(cloud))
    del base


@pytest.mark.parametrize("shape,n", [((16, 1800), 5), ((64, 2048), 6), ((5, 33), 40), ((7, 300), 60)])
def test_labels_batch_dev(pkg, ctxs, oracle, synth, shape, n):
    """Batched labelling (TMA-fed kernel when the shape allows it, plain kernel otherwise)."""
    torch = pytest.importorskip("torch")
    ctx = ctxs(shape)
    frames = np.stack([_cloud(synth, shape, f, invalid_frac=0.01 if f % 3 == 0 else 0.0) for f in range(n)])
    d_clouds = torch.from_numpy(frames).cuda()
    d_labels = torch.empty(frames.shape[:-1], dtype=torch.int32, device="cuda")
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    ctx.extract_feature_batch_dev(d_clouds.data_ptr(), frames.shape[0], d_labels.data_ptr())
    torch.cuda.synchronize()
    ctx.set_stream(None)
    got = d_labels.cpu().numpy()
    for f in range(frames.shape[0]):
        assert np.array_equal(got[f], oracle.extract_feature(frames[f]))


# ------------------------------------------------------------------ a2 / a4 / a7 -------------
@pytest.mark.parametrize("shape", [(8, 8), (5, 33), (16, 1800)])
def test_convert_bit_exact(ctxs, oracle, shape):
    rng = np.random.default_rng(11)
    d = rng.integers(-5, 4000, size=shape).astype(np.int32)
    d[0, 0] = 0
    assert np.array_equal(ctxs(shape).convert_to_pointcloud(d), oracle.convert(d))


@pytest.mark.parametrize("shape", [(5, 33), (64, 2048)])
def test_transform_bit_exact(ctxs, oracle, synth, shape):
    rng = np.random.default_rng(5)
    cloud = _cloud(synth, shape, 1)
    for _ in range(3):
        pos = np.concatenate([rng.normal(0, 5000, 3), rng.uniform(-180, 180, 3)])
        assert np.array_equal(ctxs(shape).transform_cloud(cloud, pos), oracle.transform(cloud, pos))


@pytest.mark.parametrize("shape", SHAPES)
def test_flatten_bit_exact(ctxs, oracle, synth, shape):
    cloud = _cloud(synth, shape, 1)
    feat = oracle.extract_feature(cloud)
    feat[0, 0] = 1
    feat[0, 1] = 2
    feat[-1, -1] = 1
    ctx = ctxs(shape)
    for r in (0, shape[0] - 1):
        assert np.array_equal(ctx.flatten_points(cloud[r], feat[r]), oracle.flatten(cloud[r], feat[r]))
    none = np.zeros(shape[1], dtype=np.int32)
    assert ctx.flatten_points(cloud[0], none).shape == (0, 3)
    assert np.array_equal(ctx.flatten_points(cloud[0], none + 1), cloud[0])


# ------------------------------------------------------------------ frame path (a3+a7+a4+a5+a6)
@pytest.mark.parametrize("shape,frames", [((8, 8), 6), ((5, 33), 6), ((16, 1800), 4), ((64, 2048), 3)])
def test_frontend_frames_bit_exact(ctxs, oracle, synth, shape, frames):
    r, c = shape
    ctx = ctxs(shape)
    slam = oracle.slam(r, c, 1)
    rng = np.random.default_rng(17)
    if shape == (8, 8):
        clouds = [oracle.convert(synth.l5_depth_frame(f)) for f in range(frames)]
    else:
        clouds = [_cloud(synth, shape, f, invalid_frac=0.01 if f == 2 else 0.0) for f in range(frames)]
    pos = np.array([10.0, -20.0, 5.0, 1.0, -2.0, 30.0])
    assert np.array_equal(ctx.slam_init(pos, clouds[0]), slam.init(pos, clouds[0]))
    for row in (0, r - 1):
        pts, col = ctx.row_map_export(row)
        feat0 = oracle.extract_feature(clouds[0])
        assert np.array_equal(col, np.nonzero(feat0[row] == 1)[0])
    last = pos
    for f in range(1, frames):
        pred = last + np.concatenate([rng.normal(45, 5, 1), rng.normal(0, 3, 2), rng.normal(0, 0.3, 3)])
        final = pred + np.concatenate([rng.normal(0, 2, 3), rng.normal(0, 0.05, 3)])
        feat, idx, dist, g = ctx.frontend_frame(clouds[f], pred, last, final)
        ofeat, oidx, odist, og = slam.frontend_frame(clouds[f], pred, last, final)
        assert np.array_equal(feat, ofeat)
        assert np.array_equal(idx, oidx), (f, np.nonzero(idx != oidx))
        assert np.array_equal(dist, odist)
        assert np.array_equal(g, og)
        last = final
    slam.close()


def test_frontend_empty_rows_and_no_features(ctxs, oracle):
    """Rows whose previous frame had no edge points (NULL tree in the reference) and frames with
    no labelled points at all."""
    shape = (5, 33)
    ctx = ctxs(shape)
    slam = oracle.slam(*shape, 1)
    rng = np.random.default_rng(1)
    flat = np.zeros((5, 33, 3))
    flat[..., 0] = 1000.0  # all points identical -> avg 0 -> no labels anywhere
    noisy = rng.normal(0, 1000, size=(5, 33, 3))
    z = np.zeros(6)
    assert np.array_equal(ctx.slam_init(z, flat), slam.init(z, flat))
    a = ctx.frontend_frame(noisy, z, z, z)
    b = slam.frontend_frame(noisy, z, z, z)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert (a[1] == -1).all() and np.isinf(a[2][a[0] == 1]).all()
    a = ctx.frontend_frame(flat, z, z, z)
    b = slam.frontend_frame(flat, z, z, z)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert a[0].sum() == 0
    slam.close()


def test_frontend_multi_sequence(pkg, oracle, synth):
    """n_seq sequences side by side give exactly what n_seq separate contexts give."""
    shape, n_seq = (16, 1800), 3
    ctx = pkg.Context(*shape, device=0, n_seq=n_seq)
    slams = [oracle.slam(*shape, 1) for _ in range(n_seq)]
    clouds = [np.stack([synth.room_frame(*shape, f, seq=s) for s in range(n_seq)]) for f in range(3)]
    pos0 = np.stack([np.array([100.0 * s, 0, 0, 0, 0, 1.0 * s]) for s in range(n_seq)])
    g = ctx.slam_init(pos0, clouds[0])
    for s in range(n_seq):
        assert np.array_equal(g[s], slams[s].init(pos0[s], clouds[0][s]))
    last = pos0
    for f in (1, 2):
        pred = last + np.array([50.0, 1.0, 0.0, 0.0, 0.0, 0.1])
        final = pred + np.array([0.5, -0.5, 0.1, 0.0, 0.0, 0.0])
        feat, idx, dist, g = ctx.frontend_frame(clouds[f], pred, last, final)
        for s in range(n_seq):
            ofeat, oidx, odist, og = slams[s].frontend_frame(clouds[f][s], pred[s], last[s], final[s])
            assert np.array_equal(feat[s], ofeat) and np.array_equal(idx[s], oidx)
            assert np.array_equal(dist[s], odist) and np.array_equal(g[s], og)
        last = final
    ctx.close()
    for s in slams:
        s.close()


@pytest.mark.parametrize("shape", [(8, 8), (16, 1800)])
def test_frontend_frame_from_depth(ctxs, oracle, synth, shape):
    """8f #3: depth matrix in, convertToPointCloud fused in front of the frame kernel."""
    r, c = shape
    ctx = ctxs(shape)
    slam = oracle.slam(r, c, 1)
    rng = np.random.default_rng(4)
    depth = [synth.l5_depth_frame(f, r, c) if shape == (8, 8) else
             (3000 + 40 * np.sin(np.arange(c) / 9.0)[None, :] + rng.integers(-6, 7, size=(r, c)) - 15 * f).astype(np.int32)
             for f in range(4)]
    depth[2][0, :3] = 0  # invalid returns -> (0,0,0)
    clouds = [oracle.convert(d) for d in depth]
    z = np.zeros(6)
    assert np.array_equal(ctx.slam_init(z, clouds[0]), slam.init(z, clouds[0]))
    last = z
    for f in range(1, 4):
        pred = last + np.array([-14.0, 0.5, 0.0, 0.0, 0.0, 0.1])
        final = last + np.array([-15.0, 0.0, 0.0, 0.0, 0.0, 0.0])
        cloud, feat, idx, dist, g = ctx.frontend_frame_depth(depth[f], pred, last, final)
        ofeat, oidx, odist, og = slam.frontend_frame(clouds[f], pred, last, final)
        assert np.array_equal(cloud, clouds[f]) and np.array_equal(feat, ofeat)
        assert np.array_equal(idx, oidx) and np.array_equal(dist, odist) and np.array_equal(g, og)
        last = final
    slam.close()


def test_frontend_async_pipeline_matches_sync(pkg, oracle, synth):
    """nav_frontend_frame_async (three overlapping streams, two slots) returns what the blocking call
    returns, frame for frame."""
    torch = pytest.importorskip("torch")
    shape, n = (16, 1800), 7
    r, c = shape
    ctx = pkg.Context(r, c, device=0)
    slam = oracle.slam(r, c, 1)
    clouds = torch.from_numpy(np.stack([synth.room_frame(r, c, f) for f in range(n)])).pin_memory()
    feat = torch.empty((n, r, c), dtype=torch.int32).pin_memory()
    idx = torch.empty((n, r, c), dtype=torch.int32).pin_memory()
    dist = torch.empty((n, r, c), dtype=torch.float64).pin_memory()
    glob = torch.empty((n, r, c, 3), dtype=torch.float64).pin_memory()
    pos0 = np.zeros(6)
    ctx.slam_init(pos0, clouds[0].numpy())
    slam.init(pos0, clouds[0].numpy())
    poses = []
    last = pos0
    for f in range(1, n):
        pred = last + np.array([49.0, 1.0, 0.0, 0.0, 0.0, 0.2])
        final = last + np.array([50.0, 0.0, 0.0, 0.0, 0.0, 0.0])
        poses.append((pred, last, final))
        ctx.frontend_frame_async(clouds[f].data_ptr(), pred, last, final, feat[f].data_ptr(), idx[f].data_ptr(),
                                 dist[f].data_ptr(), glob[f].data_ptr())
        last = final
    ctx.frontend_wait()
    for f in range(1, n):
        pred, last, final = poses[f - 1]
        ofeat, oidx, odist, og = slam.frontend_frame(clouds[f].numpy(), pred, last, final)
        assert np.array_equal(feat[f].numpy(), ofeat) and np.array_equal(idx[f].numpy(), oidx)
        assert np.array_equal(dist[f].numpy(), odist) and np.array_equal(glob[f].numpy(), og)
    # the blocking API continues seamlessly from the pipelined state
    pred, final = last + np.array([49.0, 0, 0, 0, 0, 0]), last + np.array([50.0, 0, 0, 0, 0, 0])
    extra = synth.room_frame(r, c, n)
    a = ctx.frontend_frame(extra, pred, last, final)
    b = slam.frontend_frame(extra, pred, last, final)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    with pytest.raises(pkg.NavError):  # pageable memory is refused
        ctx.frontend_frame_async(extra.ctypes.data, pred, last, final, None, None, None, None)
    ctx.close()
    slam.close()


# ------------------------------------------------------------------ whole step (a8 + Adam) ---
@pytest.mark.parametrize("shape,frames", [((8, 8), 8), ((5, 33), 6), ((16, 1800), 3), ((64, 2048), 2)])
def test_slam_step_bit_exact(ctxs, oracle, synth, shape, frames):
    r, c = shape
    ctx = ctxs(shape)
    slam = oracle.slam(r, c, 1)
    if shape == (8, 8):
        clouds = [oracle.convert(synth.l5_depth_frame(f)) for f in range(frames)]
    else:
        clouds = [_cloud(synth, shape, f) for f in range(frames)]
    pos = np.array([10.0, -20.0, 5.0, 1.0, -2.0, 30.0])
    assert np.array_equal(ctx.slam_init(pos, clouds[0]), slam.init(pos, clouds[0]))
    last = pos
    for f in range(1, frames):
        pred = last + np.array([45.0, 3.0, -1.0, 0.0, 0.0, 0.0])
        corr = ctx.slam_match(clouds[f], pred, last)
        p_gpu, err_gpu = ctx.slam_localization(clouds[f], pred, last)
        p_or, corr_or, err_or, _ = slam.localize(clouds[f], pred, last)
        assert corr.shape == corr_or.shape
        assert np.array_equal(corr, corr_or)
        assert np.array_equal(p_gpu, p_or) and err_gpu == err_or
        g = ctx.slam_mapping(p_gpu, None)           # reuse the resident frame
        g2 = ctx.slam_mapping(p_gpu, clouds[f])     # strict re-upload, same answer
        og = slam.map(p_or, clouds[f])
        assert np.array_equal(g, og) and np.array_equal(g2, og)
        last = p_gpu
    slam.close()


def test_localization_from_sufficient_statistics(ctxs, oracle, synth):
    """SURVEY 8f #2: the fit from five device-reduced sums agrees with the reference's sequential loop
    to rounding (tolerance parity: the summation order differs)."""
    shape = (64, 2048)
    ctx = ctxs(shape)
    slam = oracle.slam(*shape, 1)
    clouds = [synth.room_frame(*shape, f) for f in range(3)]
    pos = np.zeros(6)
    ctx.slam_init(pos, clouds[0])
    slam.init(pos, clouds[0])
    last = pos
    for f in (1, 2):
        pred = last + np.array([46.0, 2.0, -1.0, 0.0, 0.0, 0.0])
        p_fast, err_fast, n_fast = ctx.slam_localization_fast(clouds[f], pred, last)
        p_or, corr, err_or, _ = slam.localize(clouds[f], pred, last)
        assert n_fast == corr.shape[0]
        assert np.allclose(p_fast, p_or, rtol=1e-9, atol=1e-6), p_fast - p_or
        assert abs(err_fast - err_or) <= 1e-6 * max(1.0, err_or)
        ctx.slam_mapping(p_or, None)
        slam.map(p_or, clouds[f])
        last = p_or
    slam.close()


# ------------------------------------------------------------------ kd-tree (a5 / a6) --------
def _check_inorder(nodes, axes, lo, hi, depth, split):
    """Recursive invariant check of the in-order layout: left keys <= node key <= right keys along the
    node's split axis; cyclic trees split depth % 3, widest-extent trees the axis of largest extent."""
    stack = [(lo, hi, depth)]
    while stack:
        lo, hi, d = stack.pop()
        if hi - lo <= 1:
            continue
        mid = lo + (hi - lo) // 2
        a = int(axes[mid])
        if split == "cyclic":
            assert a == d % 3
        else:
            ext = nodes[lo:hi].max(axis=0) - nodes[lo:hi].min(axis=0)
            assert ext[a] == ext.max() and a == int(np.argmax(ext))
        k = nodes[mid, a]
        assert (nodes[lo:mid, a] <= k).all() and (nodes[mid + 1:hi, a] >= k).all()
        stack.append((lo, mid, d + 1))
        stack.append((mid + 1, hi, d + 1))


@pytest.mark.parametrize("split", ["widest", "cyclic"])
@pytest.mark.parametrize("kind", ["uniform", "clustered", "integer", "duplicates", "sorted", "all_equal", "planes",
                                  "tight_cluster", "integer_walls"])
@pytest.mark.parametrize("n", [0, 1, 2, 3, 17, 1000, 2049, 4096, 30000, 70001])
def test_kdtree_exact_lowest_index(pkg, oracle, synth, kind, n, split):
    rng = np.random.default_rng(n + 13)
    if kind == "tight_cluster":
        # nearly all keys inside one histogram bin of the first selection round (a few far outliers stretch the
        # box): the candidates do not fit in shared memory and the range is narrowed on the lower key bits
        pts = 1.0e6 + rng.uniform(0.0, 1.0e-3, size=(n, 3))
        if n >= 17:
            pts[rng.integers(0, n, 10)] = rng.uniform(-1.0e9, 1.0e9, size=(10, 3))
    elif kind == "integer_walls":
        # integer millimetres with two thirds of the points on walls (one coordinate equal for thousands of
        # points): equal keys beyond the shared-memory capacity, resolved on the point index
        pts = np.rint(rng.uniform(-8000, 8000, size=(n, 3)))
        if n:
            wall = rng.random(n) < 0.67
            ax = rng.integers(0, 2, n)
            pts[np.arange(n)[wall], ax[wall]] = rng.choice([-8000.0, 8000.0], int(wall.sum()))
    elif kind == "uniform":
        pts = synth.map_points(n, seed=n)
    elif kind == "clustered":
        pts = synth.map_points(n, variant="clustered", seed=n)
    elif kind == "integer":
        pts = rng.integers(0, 40, size=(n, 3)).astype(np.float64)
    elif kind == "duplicates":
        pts = np.repeat(rng.normal(0, 100, size=((n + 3) // 4, 3)), 4, axis=0)[:n]
    elif kind == "sorted":
        pts = np.stack([np.arange(n, dtype=np.float64)] * 3, axis=1)
    elif kind == "planes":  # walls: one coordinate constant per point, the case cyclic splitting handles badly
        pts = rng.uniform(-4000, 4000, size=(n, 3))
        if n:
            pts[np.arange(n), rng.integers(0, 3, n)] = rng.choice([-4000.0, 4000.0], n)
    else:
        pts = np.full((n, 3), 3.25)
    tree = pkg.KdTree(pts, device=0, split=split)
    assert len(tree) == n
    nodes, oidx, axes = tree.export(with_axes=True)
    if n:
        assert np.array_equal(np.sort(oidx), np.arange(n))
        assert np.array_equal(nodes, pts[oidx])
        _check_inorder(nodes, axes, 0, n, 0, split)
    nq = 500
    q = (pts[rng.integers(0, n, size=nq)] + rng.normal(0, 3, size=(nq, 3))) if n else rng.normal(size=(nq, 3))
    if kind in ("integer", "all_equal"):
        q = np.rint(q)
    idx, dist, near = tree.nn_batch(q)
    oi, od = oracle.nn_brute(pts, q)
    assert np.array_equal(idx, oi)
    assert np.array_equal(dist, od)
    if n:
        assert np.array_equal(near, pts[oi])
    tree.close()


def test_kdtree_same_tree_as_reference_when_keys_distinct(pkg, oracle, synth):
    """With distinct keys the median-split tree is unique, so our flat in-order array must be the
    array the reference's in-place recursion leaves behind (utils/kdtree.c:65-82)."""
    pts = synth.map_points(5000, seed=77)
    h, perm = oracle.tree_build(pts)
    oracle.tree_free(h)
    tree = pkg.KdTree(pts, device=0, split="cyclic")
    nodes, _ = tree.export()
    assert np.array_equal(nodes, perm)
    tree.close()
    # the default (widest-extent) tree is a different tree with the same answers
    wide = pkg.KdTree(pts, device=0)
    q = synth.map_queries(pts, 2000, seed=78)
    assert not np.array_equal(wide.export()[0], perm)
    cyc = pkg.KdTree(pts, device=0, split="cyclic")
    a, b = wide.nn_batch(q), cyc.nn_batch(q)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    wide.close()
    cyc.close()


def test_kdtree_special_values(pkg, oracle):
    rng = np.random.default_rng(2)
    pts = rng.normal(0, 100, size=(2000, 3))
    pts[5] = np.nan
    pts[6, 1] = np.nan
    pts[7] = np.inf
    pts[8] = -np.inf
    pts[9] = 0.0
    pts[10] = -0.0
    q = rng.normal(0, 100, size=(300, 3))
    q[0] = 0.0
    tree = pkg.KdTree(pts, device=0)
    idx, dist, _ = tree.nn_batch(q)
    oi, od = oracle.nn_brute(pts, q)
    assert np.array_equal(idx, oi) and np.array_equal(dist, od)
    tree.close()


def test_kdtree_1m_vs_bruteforce(pkg, oracle, synth):
    """Config 4 size: 1 M-point map, 131 072 queries.  Checked against the exact fp64 brute-force
    kernel on a 4096-query subset and against the CPU oracle on 64 queries; all queries must
    return a point at the reported distance."""
    torch = pytest.importorskip("torch")
    for variant, qvar in (("uniform", "jitter"), ("clustered", "uniform")):
        pts = synth.map_points(1_000_000, variant=variant)
        q = synth.map_queries(pts, 131072, variant=qvar)
        tree = pkg.KdTree(pts, device=0)
        idx, dist, near = tree.nn_batch(q)
        d_back = np.sqrt(((near - q) ** 2)[:, 0] + ((near - q) ** 2)[:, 1] + ((near - q) ** 2)[:, 2])
        assert np.array_equal(near, pts[idx])
        assert np.array_equal(d_back, dist)
        sub = slice(0, 4096)
        d_pts = torch.from_numpy(pts).cuda()
        d_q = torch.from_numpy(q[sub]).cuda()
        d_idx = torch.empty(4096, dtype=torch.int32, device="cuda")
        d_dist = torch.empty(4096, dtype=torch.float64, device="cuda")
        pkg.bruteforce_nn_dev(0, d_pts.data_ptr(), pts.shape[0], d_q.data_ptr(), 4096, d_idx.data_ptr(),
                              d_dist.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(d_idx.cpu().numpy(), idx[sub])
        assert np.array_equal(d_dist.cpu().numpy(), dist[sub])
        oi, od = oracle.nn_brute(pts, q[:64])
        assert np.array_equal(oi, idx[:64]) and np.array_equal(od, dist[:64])
        tree.close()


@pytest.mark.parametrize("kind", ["uniform", "clustered", "integer", "duplicates", "offset", "line", "special"])
@pytest.mark.parametrize("n,nq", [(1, 5), (31, 200), (256, 128), (1000, 777), (5000, 4096)])
def test_bruteforce_tensor_cores_exact(pkg, oracle, synth, kind, n, nq):
    """tcgen05 candidate tiles + exact re-rank (bf_tc.cu) must give the canonical exact answer on
    every input: same idx (lowest index on ties) and bit-identical distance as the CPU oracle."""
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(n * 7 + nq)
    if kind == "uniform":
        pts = synth.map_points(n, seed=n)
    elif kind == "clustered":
        pts = synth.map_points(n, variant="clustered", seed=n)
    elif kind == "integer":
        pts = rng.integers(0, 30, size=(n, 3)).astype(np.float64)        # many exact ties
    elif kind == "duplicates":
        pts = np.repeat(rng.normal(0, 100, size=((n + 3) // 4, 3)), 4, axis=0)[:n]
    elif kind == "offset":
        pts = rng.normal(0, 20, size=(n, 3)) + np.array([3.0e7, -2.0e7, 1.0e7])  # dense, far from the origin
    elif kind == "line":
        pts = np.stack([np.arange(n, dtype=np.float64) * 0.001] * 3, axis=1) + 5.0e4
    else:
        pts = rng.normal(0, 100, size=(n, 3))
        pts[0] = np.nan
        if n > 3:
            pts[2, 1] = np.inf
    q = pts[rng.integers(0, n, size=nq)] + rng.normal(0, 3, size=(nq, 3))
    q = np.nan_to_num(q, nan=1.0, posinf=2.0, neginf=-2.0)
    if kind == "integer":
        q = np.rint(q)
    d_pts, d_q = torch.from_numpy(pts).cuda(), torch.from_numpy(q).cuda()
    d_idx = torch.empty(nq, dtype=torch.int32, device="cuda")
    d_dist = torch.empty(nq, dtype=torch.float64, device="cuda")
    pkg.bruteforce_nn_dev(0, d_pts.data_ptr(), n, d_q.data_ptr(), nq, d_idx.data_ptr(), d_dist.data_ptr(),
                          use_tensor_cores=True, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    oi, od = oracle.nn_brute(pts, q)
    assert np.array_equal(d_idx.cpu().numpy(), oi)
    assert np.array_equal(d_dist.cpu().numpy(), od)


def test_no_device_errors_are_loud(pkg):
    with pytest.raises(pkg.NavError):
        pkg.Context(8, 8, device=99)
    with pytest.raises(pkg.NavError):
        pkg.Context(8, 8, device=0, n_seq=1000)


# ------------------------------------------------------------ 8f #4: CSV rows on the GPU ----------
@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(8, 8), (5, 33), (16, 1800), (64, 2048)])
def test_csv_rows_gpu_byte_identical_to_printf(pkg, oracle, shape):
    """nav_csv_format_frame_gpu against the oracle's snprintf restatement of src/main.c:324-349."""
    rows, cols = shape
    rng = np.random.default_rng(rows * 7 + cols)
    g = rng.standard_normal((rows, cols, 3)) * 10.0 ** rng.integers(-4, 7, (rows, cols, 1))
    k = rng.integers(0, 2 ** 20, (rows, cols, 3))
    ties = rng.random((rows, cols, 3)) < 0.3
    g = np.where(ties, (2 * k + 1) / 8.0 * rng.choice([-1.0, 1.0], (rows, cols, 3)), g)   # exact x.xx5 ties
    g[0, 0] = [0.0, -0.0, 5e-324]
    g[0, 1] = [0.005, 0.015, -0.025]
    g[0, 2] = [2.0 ** 56, -(2.0 ** 57 - 16), 99.995]
    d = rng.integers(-5000, 5000, (rows, cols)).astype(np.int32)
    lp = rng.standard_normal(6) * 1000
    ep = rng.standard_normal(6) * 1000
    imu = rng.standard_normal(6) * 1000
    ctx = pkg.Context(rows, cols)
    try:
        got = ctx.csv_rows(2 ** 33 + 5, lp, global_cloud=g, distances=d, imu=imu, ekf_pos=ep)
        want = oracle.csv_format_frame(2 ** 33 + 5, g, lp, distances=d, imu=imu, ekf_pos=ep)
        assert got == want
        got = ctx.csv_rows(0, lp, global_cloud=g)
        assert got == oracle.csv_format_frame(0, g, lp)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_csv_rows_gpu_resident_cloud_and_host_fallback(pkg, oracle, synth):
    """global_cloud=None prints the cloud nav_slam_mapping left in HBM; inf / nan / huge values take
    the host formatter and still give printf's bytes."""
    rows, cols = 16, 1800
    seq = synth.l9_sequence(2)
    pos = np.array([10.0, -20.0, 5.0, 1.0, 2.0, 3.0])
    ctx = pkg.Context(rows, cols)
    try:
        g = ctx.slam_init(pos, seq[0])
        got = ctx.csv_rows(3, pos)
        assert got == oracle.csv_format_frame(3, g, pos)
        bad = g.copy()
        bad[3, 7] = [float("inf"), float("nan"), 1e300]
        got = ctx.csv_rows(4, pos, global_cloud=bad)
        assert got == oracle.csv_format_frame(4, bad, pos)
        huge_pose = pos.copy()
        huge_pose[0] = 1e200
        got = ctx.csv_rows(5, huge_pose, global_cloud=g)
        assert got == oracle.csv_format_frame(5, g, huge_pose)
    finally:
        ctx.close()


# ------------------------------------------------- device-resident sequence replay (bench `value`) ----
def _dev_to_numpy(torch, ptr, dtype, count):
    """Copy `count` elements from a raw device pointer (results owned by the context) to numpy."""
    import ctypes
    out = np.empty(count, dtype=dtype)
    cudart = ctypes.CDLL("libcudart.so")
    rc = cudart.cudaMemcpy(ctypes.c_void_p(out.ctypes.data), ctypes.c_void_p(ptr), ctypes.c_size_t(out.nbytes),
                           ctypes.c_int(2))  # cudaMemcpyDeviceToHost
    assert rc == 0, rc
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("shape,n_seq,n_frames", [((64, 2048), 1, 12), ((16, 1800), 1, 9), ((5, 33), 1, 6),
                                                   ((16, 1800), 3, 5)])
def test_sequence_dev_matches_oracle(pkg, oracle, synth, shape, n_seq, n_frames):
    """nav_frontend_sequence_dev: one launch per frame, consecutive launches overlapped by programmatic
    dependent launch.  Stopping the replay after k frames must leave exactly what the oracle has after k
    frames (labels, NN index / distance of frame k and the mapped cloud), for several k -- a hazard
    between overlapping launches would corrupt an intermediate map and show up in a later frame."""
    torch = pytest.importorskip("torch")
    r, c = shape
    npx = r * c
    frames = np.stack([np.stack([synth.room_frame(r, c, f, seq=s) for s in range(n_seq)]) for f in range(n_frames)])
    d_frames = torch.from_numpy(frames).cuda()                      # [frame][seq][r][c][3]
    stream = torch.cuda.Stream()
    pos0 = np.zeros((n_seq, 6))
    pred = np.stack([np.stack([np.array([50.0 * f - 1.0, 1.0 + s, 0, 0, 0, 0.2]) for s in range(n_seq)])
                     for f in range(n_frames)])
    final = np.stack([np.stack([np.array([50.0 * f, 0.5 * s, 0, 0, 0, 0.0]) for s in range(n_seq)])
                      for f in range(n_frames)])
    last = np.concatenate([pos0[None], final[:-1]])
    slams = [oracle.slam(r, c, 1) for _ in range(n_seq)]
    for s in range(n_seq):
        slams[s].init(pos0[s], frames[0, s])
    want = {}
    for f in range(1, n_frames):
        want[f] = [slams[s].frontend_frame(frames[f, s], pred[f, s], last[f, s], final[f, s]) for s in range(n_seq)]
    ctx = pkg.Context(r, c, device=0, n_seq=n_seq)
    try:
        ctx.set_stream(stream.cuda_stream)
        for k in sorted({1, 2, n_frames // 2, n_frames - 1}):
            ctx.slam_init_dev(d_frames[0].data_ptr(), pos0)
            ctx.frontend_sequence_dev(d_frames[1].data_ptr(), k, pred[1:k + 1].reshape(-1, 6),
                                      last[1:k + 1].reshape(-1, 6), final[1:k + 1].reshape(-1, 6))
            stream.synchronize()
            res = ctx.frame_results_dev()

            labels = _dev_to_numpy(torch, res.labels, np.int32, n_seq * npx).reshape(n_seq, r, c)
            idx = _dev_to_numpy(torch, res.nn_idx, np.int32, n_seq * npx).reshape(n_seq, r, c)
            dist = _dev_to_numpy(torch, res.nn_dist, np.float64, n_seq * npx).reshape(n_seq, r, c)
            glob = _dev_to_numpy(torch, res.global_, np.float64, n_seq * npx * 3).reshape(n_seq, r, c, 3)
            for s in range(n_seq):
                ofeat, oidx, odist, og = want[k][s]
                lab = ofeat == 1
                assert np.array_equal(labels[s], ofeat), (k, s)
                assert np.array_equal(idx[s][lab], oidx[lab]) and np.array_equal(dist[s][lab], odist[lab]), (k, s)
                assert np.array_equal(glob[s], og), (k, s)
    finally:
        ctx.close()
        for sl in slams:
            sl.close()


# ------------------------------------------------- odd shapes: every search path of the frame kernel ----
@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 5), (2, 17), (3, 255), (3, 256), (3, 257), (2, 513), (2, 2049), (2, 4100),
                                   (1, 14000)])
@pytest.mark.parametrize("motion", ["small", "large", "scrambled"])
def test_frontend_frame_odd_shapes(pkg, oracle, synth, shape, motion):
    """Widths around the 16 / 256-column block sizes, rows wider than the shared-memory copy of the leaf
    boxes (> 2048 columns; nav_create caps rows at about 14 500 columns), and motions that send queries far
    from their own column ('large': 30 degrees of yaw; 'scrambled': the previous frame's columns are
    permuted, so the nearest neighbour sits in an arbitrary leaf of the row)."""
    r, c = shape
    rng = np.random.default_rng(r * 100003 + c)
    f0 = synth.room_frame(r, c, 0)
    f1 = synth.room_frame(r, c, 1)
    if motion == "scrambled":
        f0 = np.ascontiguousarray(f0[:, rng.permutation(c)])
    ctx = pkg.Context(r, c, device=0)
    slam = oracle.slam(r, c, 1)
    try:
        z = np.zeros(6)
        assert np.array_equal(ctx.slam_init(z, f0), slam.init(z, f0))
        pred = np.array([50.0, 3.0, -2.0, 0.0, 0.0, 30.0 if motion == "large" else 0.3])
        final = np.array([51.0, 2.0, -1.0, 0.1, 0.0, 0.2])
        for cloud in (f1, synth.room_frame(r, c, 2, invalid_frac=0.02)):
            a = ctx.frontend_frame(cloud, pred, z, final)
            b = slam.frontend_frame(cloud, pred, z, final)
            for x, y in zip(a, b):
                assert np.array_equal(x, y)
    finally:
        ctx.close()
        slam.close()


@pytest.mark.gpu
def test_sequence_dev_on_legacy_default_stream(pkg, oracle, synth):
    """The sequence replay also works on the legacy default stream (no programmatic dependent launch there)."""
    torch = pytest.importorskip("torch")
    r, c, n = 5, 33, 5
    frames = np.stack([synth.room_frame(r, c, f) for f in range(n)])
    d_frames = torch.from_numpy(frames).cuda()
    z = np.zeros(6)
    pred = np.stack([np.array([50.0 * f - 1.0, 1.0, 0, 0, 0, 0.2]) for f in range(n)])
    final = np.stack([np.array([50.0 * f, 0.0, 0, 0, 0, 0.0]) for f in range(n)])
    last = np.concatenate([z[None], final[:-1]])
    slam = oracle.slam(r, c, 1)
    slam.init(z, frames[0])
    for f in range(1, n):
        want = slam.frontend_frame(frames[f], pred[f], last[f], final[f])
    ctx = pkg.Context(r, c, device=0)
    try:
        ctx.set_stream(0)
        torch.cuda.synchronize()
        ctx.slam_init_dev(d_frames[0].data_ptr(), z)
        ctx.frontend_sequence_dev(d_frames[1].data_ptr(), n - 1, pred[1:], last[1:], final[1:])
        torch.cuda.synchronize()
        res = ctx.frame_results_dev()
        labels = _dev_to_numpy(torch, res.labels, np.int32, r * c).reshape(r, c)
        idx = _dev_to_numpy(torch, res.nn_idx, np.int32, r * c).reshape(r, c)
        glob = _dev_to_numpy(torch, res.global_, np.float64, r * c * 3).reshape(r, c, 3)
        lab = want[0] == 1
        assert np.array_equal(labels, want[0]) and np.array_equal(idx[lab], want[1][lab]) and np.array_equal(glob, want[3])
    finally:
        ctx.close()
        slam.close()


# ------------------------------------------------------------------ round 2 additions --------
@pytest.mark.gpu
@pytest.mark.parametrize("shape,n", [((5, 33), 1001), ((3, 67), 1501), ((5, 33), 1000)])
def test_labels_batch_odd_point_count_takes_the_tma_path(pkg, oracle, shape, n):
    """A batch with an ODD number of points ends in a tile whose byte count is 8 mod 16, which a bulk copy
    cannot move (sizes must be multiples of 16): the producer stores the trailing double itself.  The batch
    is large enough (>= 4 tiles per SM) for launch_labels to choose k_labels_tma."""
    torch = pytest.importorskip("torch")
    r, c = shape
    rng = np.random.default_rng(r * 1000 + c + n)
    base = np.cumsum(rng.normal(0, 30, size=(n, r, c, 3)), axis=2)  # rough polylines: a healthy mix of labels
    assert (n * r * c) % 2 == (n % 2)
    ctx = pkg.Context(r, c, device=0)
    d = torch.from_numpy(base).cuda()
    lab = torch.full((n, r, c), -7, dtype=torch.int32, device="cuda")
    ctx.extract_feature_batch_dev(d.data_ptr(), n, lab.data_ptr())
    torch.cuda.synchronize()
    got = lab.cpu().numpy()
    for i in list(range(0, n, max(n // 23, 1))) + [n - 1, n - 2]:   # the last images hold the odd tail
        assert np.array_equal(got[i], oracle.extract_feature(base[i])), i
    assert set(np.unique(got)) <= {0, 1}
    ctx.close()


@pytest.mark.gpu
def test_async_wait_brings_all_results_back_into_the_context(pkg, oracle, synth):
    """After nav_frontend_wait the device-resident results (nav_frame_results_dev) are those of the last
    pipelined frame: labels AND nn_idx / nn_dist (round-1 advisor finding)."""
    torch = pytest.importorskip("torch")
    r, c, n = 16, 1800, 4
    ctx = pkg.Context(r, c, device=0)
    clouds = torch.from_numpy(np.stack([synth.room_frame(r, c, f) for f in range(n)])).pin_memory()
    outs = [torch.empty(r * c * 16, dtype=torch.uint8).pin_memory() for _ in range(2)]
    z = np.zeros(6)
    ctx.slam_init(z, clouds[0].numpy())
    last = z
    for f in range(1, n):
        final = last + np.array([50.0, 0, 0, 0, 0, 0])
        p0 = outs[f & 1].data_ptr()
        ctx.frontend_frame_async(clouds[f].data_ptr(), final + 1.0, last, final, p0, p0 + r * c * 4, p0 + r * c * 8, None)
        last = final
    ctx.frontend_wait()
    res = ctx.frame_results_dev()
    host = outs[(n - 1) & 1].numpy()
    # wrap the context's raw device pointers for torch through the CUDA array interface
    class Raw:
        def __init__(self, ptr, n, typestr):
            self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}
    lab = torch.as_tensor(Raw(res.labels, r * c, "<i4"), device="cuda").cpu().numpy()
    idx = torch.as_tensor(Raw(res.nn_idx, r * c, "<i4"), device="cuda").cpu().numpy()
    dist = torch.as_tensor(Raw(res.nn_dist, r * c, "<f8"), device="cuda").cpu().numpy()
    assert np.array_equal(lab, host[: r * c * 4].view(np.int32))
    assert np.array_equal(idx, host[r * c * 4: r * c * 8].view(np.int32))
    assert np.array_equal(dist, host[r * c * 8:].view(np.float64))
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(8, 8), (16, 1800), (5, 33)])
def test_submit_depth_input_and_label_masks(pkg, oracle, synth, shape):
    """nav_frontend_submit with the L5 depth matrix as input (utils/pointcloud.c:8 on the device) and the
    labels returned as 16-bit masks: same labels / NN / clouds as the oracle, frame for frame, pipelined."""
    torch = pytest.importorskip("torch")
    r, c = shape
    n = 6
    ctx = pkg.Context(r, c, device=0)
    slam = oracle.slam(r, c, 1)
    rng = np.random.default_rng(r + c)
    depth = np.stack([(3000 + 40 * np.sin(np.arange(c) / 9.0)[None, :] + rng.integers(-6, 7, size=(r, c)) - 15 * f)
                      for f in range(n)]).astype(np.int32)
    depth[2, 0, :3] = 0
    clouds = [oracle.convert(d) for d in depth]
    h_depth = torch.from_numpy(depth).pin_memory()
    nch = (c + 15) // 16
    mask = torch.zeros((n, r, nch), dtype=torch.int32).pin_memory()
    idx = torch.empty((n, r, c), dtype=torch.int32).pin_memory()
    dist = torch.empty((n, r, c), dtype=torch.float64).pin_memory()
    feat = torch.empty((n, r, c), dtype=torch.int32).pin_memory()
    glob = torch.empty((n, r, c, 3), dtype=torch.float64).pin_memory()
    conv = torch.empty((n, r, c, 3), dtype=torch.float64).pin_memory()
    z = np.zeros(6)
    ctx.slam_init(z, clouds[0])
    slam.init(z, clouds[0])
    poses, last = [], z
    for f in range(1, n):
        pred = last + np.array([-14.0, 0.5, 0.0, 0.0, 0.0, 0.1])
        final = last + np.array([-15.0, 0.0, 0.0, 0.0, 0.0, 0.0])
        poses.append((pred, last, final))
        kw = dict(distances=h_depth[f].data_ptr(), mask_out=mask[f].data_ptr(), nn_idx_out=idx[f].data_ptr(),
                  nn_dist_out=dist[f].data_ptr())
        if f % 2:   # odd frames ask for everything, even frames for the compact set only
            kw.update(feature_out=feat[f].data_ptr(), global_out=glob[f].data_ptr(), cloud_out=conv[f].data_ptr())
        ctx.frontend_submit(pred, last, final, **kw)
        last = final
    ctx.frontend_wait()
    for f in range(1, n):
        ofeat, oidx, odist, og = slam.frontend_frame(clouds[f], *poses[f - 1])
        m = mask[f].numpy().view(np.uint32)
        bits = ((m[:, :, None] >> np.arange(16, dtype=np.uint32)) & 1).reshape(r, nch * 16)[:, :c]
        assert np.array_equal(bits.astype(np.int32), ofeat), f
        assert np.array_equal(idx[f].numpy(), oidx) and np.array_equal(dist[f].numpy(), odist)
        if f % 2:
            assert np.array_equal(feat[f].numpy(), ofeat) and np.array_equal(glob[f].numpy(), og)
            assert np.array_equal(conv[f].numpy(), clouds[f])
    with pytest.raises(pkg.NavError):   # exactly one input
        ctx.frontend_submit(z, z, z, nn_idx_out=idx[0].data_ptr())
    ctx.close()
    slam.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shape,frames,use_depth", [((64, 2048), 6, False), ((16, 1800), 8, False), ((8, 8), 8, True)])
def test_closed_loop_with_prefetch_equals_blocking_loop(pkg, oracle, synth, shape, frames, use_depth):
    """nav_slam_prefetch + nav_slam_localization_fast + nav_slam_mapping(NULL, NULL) with pose feedback: the
    poses are bit-identical to the same loop without prefetch (the statistics are summed in a fixed order),
    agree with the reference's sequential Adam loop to rounding, and the final map equals the oracle's."""
    torch = pytest.importorskip("torch")
    r, c = shape
    if use_depth:
        depth = np.stack([synth.l5_depth_frame(f, r, c) for f in range(frames)])
        clouds = np.stack([oracle.convert(d) for d in depth])
        h_depth = torch.from_numpy(depth).pin_memory()
    else:
        clouds = np.stack([synth.room_frame(r, c, f) for f in range(frames)])
    h = torch.from_numpy(clouds).pin_memory()
    step = np.array([-19.0, 0.3, 0.0, 0, 0, 0]) if use_depth else np.array([46.0, 2.0, -1.0, 0.0, 0.0, 0.0])

    def run(prefetch):
        ctx = pkg.Context(r, c, device=0)
        ctx.slam_init(np.zeros(6), clouds[0], want_global=False)
        poses, last = [], np.zeros(6)
        def pf(f):
            if use_depth:
                ctx.slam_prefetch(depth_ptr=h_depth[f].data_ptr())
            else:
                ctx.slam_prefetch(cloud_ptr=h[f].data_ptr())
        if prefetch:
            pf(1)
        for f in range(1, frames):
            if prefetch and f + 1 < frames:
                pf(f + 1)
            if prefetch:
                p, err, n = ctx.slam_localization_fast_ptr(None if use_depth else h[f].data_ptr(), last + step, last)
            else:
                p, err, n = ctx.slam_localization_fast(clouds[f], last + step, last)
            ctx.slam_mapping(p, None, want_global=False)
            poses.append((p, err, n))
            last = p
        g = ctx.slam_mapping(last, None)   # same pose again: downloads the final map
        ctx.close()
        return poses, g

    a, ga = run(True)
    b, gb = run(False)
    for (pa, ea, na), (pb, eb, nb) in zip(a, b):
        assert np.array_equal(pa, pb) and ea == eb and na == nb
    assert np.array_equal(ga, gb)
    # the same loop as ONE call (nav_slam_run, prediction = last + step): same poses, same final map
    ctx = pkg.Context(r, c, device=0)
    ctx.slam_init(np.zeros(6), clouds[0], want_global=False)
    src = h_depth if use_depth else h
    poses, errs, ncs = ctx.slam_run([src[f].data_ptr() for f in range(1, frames)], np.tile(step, (frames - 1, 1)),
                                    np.zeros(6), depth_input=use_depth)
    for f in range(frames - 1):
        assert np.array_equal(poses[f], a[f][0]) and errs[f] == a[f][1] and ncs[f] == a[f][2]
    assert np.array_equal(ctx.slam_mapping(poses[-1], None), ga)
    ctx.close()
    slam = oracle.slam(r, c, 1)
    slam.init(np.zeros(6), clouds[0])
    last = np.zeros(6)
    for f in range(1, frames):
        p_or, corr, err_or, _ = slam.localize(clouds[f], last + step, last)
        assert a[f - 1][2] == corr.shape[0]
        assert np.allclose(a[f - 1][0], p_or, rtol=1e-9, atol=1e-6)
        og = slam.map(a[f - 1][0], clouds[f])   # feed OUR pose back so that the maps stay comparable bit for bit
        last = a[f - 1][0]
    assert np.array_equal(ga, og)
    slam.close()


@pytest.mark.gpu
def test_slam_run_with_a_prediction_callback_and_registered_memory(pkg, synth):
    """nav_slam_run driven by a caller's prediction callback (the EKF's place, src/main.c:303-306) on frames that
    live in ordinary numpy memory page-locked with nav_host_register: same poses as the array-of-increments
    form on torch-pinned memory; unpinned frames are refused."""
    import ctypes as C
    torch = pytest.importorskip("torch")
    r, c, n = 16, 1800, 6
    clouds = np.stack([synth.room_frame(r, c, f) for f in range(n)])
    step = np.array([46.0, 2.0, -1.0, 0.0, 0.0, 0.0])
    L = pkg.load_library()
    binding = __import__("importlib").import_module("nav-slam_b200.binding")
    NavPos = binding.NavPos
    ctx = pkg.Context(r, c, device=0)
    ctx.slam_init(np.zeros(6), clouds[0], want_global=False)
    h = torch.from_numpy(clouds).pin_memory()
    want, errs, ncs = ctx.slam_run([h[f].data_ptr() for f in range(1, n)], np.tile(step, (n - 1, 1)), np.zeros(6))
    # the same through a callback, frames in registered numpy memory
    own = clouds.copy()
    assert L.nav_host_register(own.ctypes.data, own.nbytes) == 0
    calls = []
    PRED = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(NavPos), C.POINTER(NavPos))

    def predict(user, t, last, pred):
        calls.append(t)
        for k, name in enumerate(("x", "y", "z", "roll", "pitch", "yaw")):
            setattr(pred[0], name, getattr(last[0], name) + step[k])
    cb = PRED(predict)
    ctx.slam_init(np.zeros(6), clouds[0], want_global=False)
    ptrs = (C.c_void_p * (n - 1))(*[own[f].ctypes.data for f in range(1, n)])
    out = (NavPos * (n - 1))()
    start = NavPos(0, 0, 0, 0, 0, 0)
    # the library handle is shared by the whole process: the callback signature is restored afterwards, so that
    # later Context.slam_run calls (predict = NULL) keep the binding's own argument types
    saved = L.nav_slam_run.argtypes
    L.nav_slam_run.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int, C.c_int, PRED, C.c_void_p, C.c_void_p,
                               C.POINTER(NavPos), C.POINTER(NavPos), C.c_void_p, C.c_void_p]
    try:
        rc = L.nav_slam_run(ctx.h, ptrs, n - 1, 0, cb, None, None, C.byref(start), out, None, None)
        assert rc == 0, L.nav_last_error()
        assert calls == list(range(n - 1))
        got = np.array([[p.x, p.y, p.z, p.roll, p.pitch, p.yaw] for p in out])
        assert np.array_equal(got, want)
        assert L.nav_host_unregister(own.ctypes.data) == 0
        # pageable frames: refused with a message, nothing queued
        ctx.slam_init(np.zeros(6), clouds[0], want_global=False)
        rc = L.nav_slam_run(ctx.h, ptrs, n - 1, 0, cb, None, None, C.byref(start), out, None, None)
        assert rc != 0 and b"pinned" in L.nav_last_error()
    finally:
        L.nav_slam_run.argtypes = saved
    ctx.close()


@pytest.mark.gpu
def test_long_sequence_launch_equals_per_frame_launches(pkg, synth):
    """70 frames in one nav_frontend_sequence_dev call (longer than the 64 frames whose poses fit the kernel
    parameters: the poses are uploaded) leave exactly what 70 nav_frontend_frame_dev calls leave -- labels, NN of the
    last frame, final map -- and the same again on a second run (no race between the tiles of a row's cluster)."""
    torch = pytest.importorskip("torch")
    r, c, n = 16, 1800, 71
    frames = np.stack([synth.room_frame(r, c, f % 23) for f in range(n)])     # 23 distinct frames, back and forth
    d_frames = torch.from_numpy(frames).cuda()
    stream = torch.cuda.Stream()
    pose = lambda f: np.array([50.0 * (f % 23), 0.3 * (f % 5), 0, 0, 0, 0.1 * (f % 3)])
    final = np.stack([pose(f) for f in range(n)])
    last = np.concatenate([np.zeros((1, 6)), final[:-1]])
    pred = final + np.array([-1.5, 0.7, 0.2, 0, 0, 0.05])
    ctx = pkg.Context(r, c, device=0)
    ctx.set_stream(stream.cuda_stream)
    npx = r * c

    def grab():
        stream.synchronize()
        res = ctx.frame_results_dev()
        return (_dev_to_numpy(torch, res.labels, np.int32, npx), _dev_to_numpy(torch, res.nn_idx, np.int32, npx),
                _dev_to_numpy(torch, res.nn_dist, np.float64, npx), _dev_to_numpy(torch, res.global_, np.float64, npx * 3))
    runs = []
    for rep in range(2):
        ctx.slam_init_dev(d_frames[0].data_ptr(), np.zeros(6))
        ctx.frontend_sequence_dev(d_frames[1].data_ptr(), n - 1, pred[1:], last[1:], final[1:])
        runs.append(grab())
    ctx.slam_init_dev(d_frames[0].data_ptr(), np.zeros(6))
    for f in range(1, n):
        ctx.frontend_frame_dev(d_frames[f].data_ptr(), pred[f], last[f], final[f])
    want = grab()
    for got in runs:
        lab = want[0] == 1
        assert np.array_equal(got[0], want[0])
        assert np.array_equal(got[1][lab], want[1][lab]) and np.array_equal(got[2][lab], want[2][lab])
        assert np.array_equal(got[3], want[3])
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["uniform", "room"])
def test_kdtree_build_is_deterministic(pkg, synth, kind):
    """The build places elements with atomic counters, but the node of a range is a function of the SET of points in
    it: repeated builds give the same node array bit for bit (uniform points; a map of plane surfaces, which takes the
    second selection round and the two-level counting sort)."""
    if kind == "uniform":
        pts = synth.map_points(300000, seed=3)
    else:
        pts, _ = synth.accumulated_map(2, rows=64, cols=2048)
    first = None
    for rep in range(3):
        tree = pkg.KdTree(pts, device=0)
        nodes, oidx, axes = tree.export(with_axes=True)
        tree.close()
        if first is None:
            first = (nodes, oidx, axes)
            assert np.array_equal(np.sort(oidx), np.arange(pts.shape[0]))
            _check_inorder(nodes, axes, 0, pts.shape[0], 0, "widest")
        else:
            assert np.array_equal(nodes, first[0]) and np.array_equal(oidx, first[1]) and np.array_equal(axes, first[2])
