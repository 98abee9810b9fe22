"""The closed loop's fit statistics against exact sums.

nav_slam_localization_fast and nav_slam_run fit the pose from five totals {N, sum r, sum |r|^2} that the device
reduces over the dedupe winners (r = ori - nearest).  Here those totals (nav_slam_fit_stats) are held to
math.fsum of the oracle's correspondence list within the error bound of the device's fixed summation tree --
exactly, where every r is an integer --, the pose to a line-by-line restatement of the host fit, and the map to
the oracle's map from the device's pose.  The cases cover every cluster width of the statistics kernels, rows
wider than 2048 columns (k_dedupe_rows), matches across the CTAs of a cluster, distance ties, degenerate
frames, and the closed-loop calls mixed with the other entry points on one context."""
import contextlib
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

STEP = np.array([46.0, 2.0, -1.0, 0.0, 0.0, 0.0])
U = 2.0 ** -53


# ------------------------------------------------------------------ helpers ----------------------------------
def exact_stats(corr):
    """N, the correctly rounded sums {rx, ry, rz, |r|^2} and the sums of their magnitudes, from the oracle's
    correspondence list (columns ori xyz | nearest xyz | distance).  r and |r|^2 are rounded as the device
    rounds them: r = ori - nearest, |r|^2 = (rx*rx + ry*ry) + rz*rz."""
    r = corr[:, 0:3] - corr[:, 3:6]
    q = (r[:, 0] * r[:, 0] + r[:, 1] * r[:, 1]) + r[:, 2] * r[:, 2]
    sums = [math.fsum(r[:, k]) for k in range(3)] + [math.fsum(q)]
    mags = [math.fsum(np.abs(r[:, k])) for k in range(3)] + [math.fsum(q)]
    return corr.shape[0], sums, mags


def sum_depth(rows, cols):
    """The most roundings any one term passes through in the device's summation tree.
    cols <= 2048 (k_dedupe_stats, k_loop_step): a 256-column tile CTA adds its column values with a 5-level
    shuffle tree, then its 8 warp partials one after another; the last CTA adds the rows*tiles CTA partials
    thread-strided (ceil(parts/256) each), with a 5-level shuffle tree, then 8 warp partials in turn.  That is
    26 + ceil(parts/256): 28 at 64x2048.
    cols > 2048 (k_dedupe_rows): a 512-thread row CTA adds ceil(cols/512) column values per thread, a 5-level
    shuffle tree, 16 warp partials in turn; the last CTA adds the row totals the same way.  At 2x4100 that is
    52, at 1x14000 71.
    The order-free bound (depth N) would let a wrong dedupe winner through on a 10^4-point frame."""
    if cols <= 2048:
        parts = rows * -(-cols // 256)
        return 5 + 8 + -(-parts // 256) + 5 + 8
    return -(-cols // 512) + 5 + 16 + -(-rows // 512) + 5 + 16


def gamma(d):
    return d * U / (1 - d * U)


def check_stats(st, corr, shape, exact=False):
    n, sums, mags = exact_stats(corr)
    assert st[0] == n
    if exact:    # every term an integer: the sums are exact whatever the order
        assert list(st[1:]) == sums, (st, sums)
        return
    # +1: fsum itself is within u*sum|x| of the exact sum
    g = gamma(sum_depth(*shape) + 1)
    for k in range(4):
        assert abs(st[1 + k] - sums[k]) <= g * mags[k], (k, st[1 + k], sums[k], g * mags[k])


_C1 = [1 - math.pow(0.9, i + 1) for i in range(200)]
_C2 = [1 - math.pow(0.999, i + 1) for i in range(200)]


def fit_py(st, pred, last):
    """fit_from_stats (csrc/capi.cu) line by line in binary64; the host code is built without contraction, so
    the bits agree.  Returns (pose, rms error, n_corr)."""
    lr, tol, b1, b2, eps = 0.1, 1e-6, 0.9, 0.999, 1e-8
    N, S, Q = float(st[0]), [float(s) for s in st[1:4]], float(st[4])
    t = [float(pred[k]) - float(last[k]) for k in range(6)]
    m, v = [0.0, 0.0, 0.0], [0.0, 0.0, 0.0]
    prev = total = 0.0
    for it in range(200):
        total = Q - 2.0 * (t[0] * S[0] + t[1] * S[1] + t[2] * S[2]) + N * (t[0] * t[0] + t[1] * t[1] + t[2] * t[2])
        if N == 0:
            total = 0.0
        if abs(total - prev) < tol:
            break
        prev = total
        for j in range(3):
            g = -(S[j] - N * t[j]) / N if N > 0 else 0.0
            m[j] = b1 * m[j] + (1 - b1) * g
            v[j] = b2 * v[j] + (1 - b2) * g * g
            mh, vh = m[j] / _C1[it], v[j] / _C2[it]
            t[j] -= lr * mh / (math.sqrt(vh) + eps)
    err = math.sqrt(max(total, 0.0) / N) if N > 0 else 0.0
    return np.array([float(last[k]) + t[k] for k in range(6)]), err, int(N)


def check_fit(st, pred, last, pose, err, n_corr):
    want, want_err, want_n = fit_py(st, pred, last)
    assert np.array_equal(pose, want), pose - want
    assert err == want_err and n_corr == want_n


@contextlib.contextmanager
def pinned(pkg, *arrays):
    """Page-lock numpy arrays in place (nav_host_register) for the calls that need pinned host memory."""
    L = pkg.load_library()
    done = []
    try:
        for a in arrays:
            assert a.flags.c_contiguous
            assert L.nav_host_register(a.ctypes.data, a.nbytes) == 0, L.nav_last_error()
            done.append(a)
        yield
    finally:
        for a in done:
            L.nav_host_unregister(a.ctypes.data)


def ptr(a):
    return a.ctypes.data


def loop_frames(synth, shape, motion, n):
    r, c = shape
    frames = np.stack([synth.room_frame(r, c, f) for f in range(n)])
    if motion == "scrambled":   # matches land in arbitrary tiles: posts across the whole cluster
        rng = np.random.default_rng(r * 7919 + c)
        for f in range(n):
            frames[f] = frames[f][:, rng.permutation(c)]
    return frames


def motion_step(motion):
    return STEP + np.array([0, 0, 0, 0, 0, 30.0]) if motion == "large" else STEP


# ------------------------------------------------------------------ every cluster width, wide rows --------------
# cluster widths 1, 1, 2, 3, 4, 5, 6, 7, 8, 8, then rows wider than 2048 columns (k_dedupe_rows + mailbox)
SHAPES = [(1, 5), (3, 256), (3, 257), (2, 600), (2, 1000), (2, 1100), (2, 1500), (2, 1700), (16, 1800), (64, 2048),
          (2, 2049), (2, 4100), (1, 14000)]
CASES = [(s, m) for s in SHAPES for m in ("small", "large", "scrambled") if s != (64, 2048)] + [((64, 2048), "small")]


@pytest.mark.parametrize("shape,motion", CASES)
def test_fit_statistics_exact_every_cluster_width(pkg, oracle, synth, shape, motion):
    r, c = shape
    n = 4
    frames = loop_frames(synth, shape, motion, n)
    step = motion_step(motion)
    z = np.zeros(6)
    slam = oracle.slam(r, c, 1)
    ctx = pkg.Context(r, c, device=0)
    with pinned(pkg, frames):
        try:
            assert np.array_equal(ctx.slam_init(z, frames[0]), slam.init(z, frames[0]))
            with pytest.raises(pkg.NavError):   # no fit yet
                ctx.slam_fit_stats()
            # separate calls: prefetch + localization_fast + mapping(NULL), statistics after every frame
            got, last = [], z
            ctx.slam_prefetch(cloud_ptr=ptr(frames[1]))
            for f in range(1, n):
                if f + 1 < n:
                    ctx.slam_prefetch(cloud_ptr=ptr(frames[f + 1]))
                pred = last + step
                p, err, nc = ctx.slam_localization_fast_ptr(ptr(frames[f]), pred, last)
                st = ctx.slam_fit_stats()
                _, corr, _, _ = slam.localize(frames[f], pred, last)
                assert nc == corr.shape[0]
                check_stats(st, corr, shape)
                check_fit(st, pred, last, p, err, nc)
                # the oracle maps the frame from the device's pose: the maps stay comparable bit for bit
                assert np.array_equal(ctx.slam_mapping(p, None), slam.map(p, frames[f]))
                got.append((p, err, nc, st))
                last = p
            # the same frames as one nav_slam_run on a fresh context
            ctx.close()
            ctx = pkg.Context(r, c, device=0)
            ctx.slam_init(z, frames[0], want_global=False)
            poses, errs, ncs = ctx.slam_run([ptr(frames[f]) for f in range(1, n)], np.tile(step, (n - 1, 1)), z)
            for f in range(n - 1):
                assert np.array_equal(poses[f], got[f][0]) and errs[f] == got[f][1] and ncs[f] == got[f][2]
            # k_loop_step sums in the order of k_dedupe_stats: the same bits
            assert np.array_equal(ctx.slam_fit_stats(), got[-1][3])
        finally:
            ctx.close()
            slam.close()


# ------------------------------------------------------------------ ties, exact integer sums ----------------
def tie_frames(synth, shape):
    """A map frame A (integer mm, even coordinates) and a query frame B built from it so that ties are certain:
    row 0: columns 2k and 2k+1 sit at A[2k] +- d (two queries at equal distance from one map point, adjacent);
    row 1: columns j and j + cols//2 sit at A[j] +- d (the same, in different tiles of the row);
    row 2: column j sits halfway between A[j] and A[j+1] (two map points at equal distance from one query)."""
    r, c = shape
    A = synth.room_frame(r, c, 0, integer_mm=True)
    A -= np.mod(A, 2.0)
    d = np.array([0.0, 0.0, 3.0])
    B = A.copy()
    j = np.arange(c)
    B[0] = A[0, j & ~1] + np.where(j % 2 == 0, 1.0, -1.0)[:, None] * d
    h = c // 2
    B[1, :h] = A[1, :h] + d
    B[1, h:2 * h] = A[1, :h] - d
    B[2, :-1] = (A[2, :-1] + A[2, 1:]) / 2
    B[2, -1] = A[2, -1] + d
    return A, B


def tie_census(oracle, A, B):
    """(map points won by one of several queries at equal distance with different positions,
        queries with several distinct map points at the least distance)."""
    la, lb = oracle.extract_feature(A), oracle.extract_feature(B)
    shared = split = 0
    for row in range(A.shape[0]):
        M = A[row][la[row] == 1]
        if len(M) == 0:
            continue
        best = {}
        for cq in np.nonzero(lb[row] == 1)[0]:
            dsq = ((M - B[row, cq]) ** 2).sum(1)
            k = np.nonzero(dsq == dsq.min())[0]
            split += len(np.unique(M[k], axis=0)) > 1
            best.setdefault(k[0], []).append((dsq.min(), cq))
        for lst in best.values():
            dmin = min(x[0] for x in lst)
            shared += len(np.unique(B[row, [cq for dq, cq in lst if dq == dmin]], axis=0)) > 1
    return shared, split


@pytest.mark.parametrize("shape", [(3, 256), (3, 300), (3, 1100), (3, 2048), (3, 4100)])   # clusters 1, 2, 5, 8; rows
def test_fit_statistics_ties_bit_exact(pkg, oracle, synth, shape):
    """Zero pose at init, integer translation and no rotation in the prediction: R is the identity, every r an
    integer, and N, sum r and sum |r|^2 are exact -- a different winner of any tie changes them."""
    r, c = shape
    A, B = tie_frames(synth, shape)
    shared, split = tie_census(oracle, A, B)
    assert shared >= c // 8 and split >= c // 8, (shared, split)
    z = np.zeros(6)
    pred = np.array([46.0, 2.0, -1.0, 0.0, 0.0, 0.0])
    slam = oracle.slam(r, c, 1)
    ctx = pkg.Context(r, c, device=0)
    with pinned(pkg, B):
        try:
            ctx.slam_init(z, A, want_global=False)
            slam.init(z, A)
            ctx.slam_prefetch(cloud_ptr=ptr(B))
            p, err, nc = ctx.slam_localization_fast_ptr(ptr(B), pred, z)
            st = ctx.slam_fit_stats()
            _, corr, _, _ = slam.localize(B, pred, z)
            check_stats(st, corr, shape, exact=True)
            check_fit(st, pred, z, p, err, nc)
            assert np.array_equal(ctx.slam_mapping(p, None), slam.map(p, B))
            # re-initialised so that the pose is an integer again: the same frame pair through nav_slam_run
            ctx.slam_init(z, A, want_global=False)
            poses, errs, ncs = ctx.slam_run([ptr(B)], pred[None], z)
            assert np.array_equal(poses[0], p) and errs[0] == err and ncs[0] == nc
            assert np.array_equal(ctx.slam_fit_stats(), st)
        finally:
            ctx.close()
            slam.close()


# ------------------------------------------------------------------ degenerate frames ------------------------
def test_fit_statistics_empty_maps_and_no_labels(pkg, oracle):
    """A previous frame without labels (every row's map empty) and a frame without labels: N = 0, all sums 0,
    and the pose is the prediction as the fit leaves it.  The reference reads uninitialised memory for queries
    against an empty row; the oracle, like the library, makes no correspondence there."""
    shape = (5, 33)
    r, c = shape
    rng = np.random.default_rng(1)
    flat = np.zeros((r, c, 3))
    flat[..., 0] = 1000.0   # all points identical: no labels anywhere
    noisy = rng.normal(0, 1000, size=(r, c, 3))
    z = np.zeros(6)
    pred = np.array([5.0, -3.0, 1.0, 0.5, 0.0, 2.0])
    slam = oracle.slam(r, c, 1)
    ctx = pkg.Context(r, c, device=0)
    try:
        assert np.array_equal(ctx.slam_init(z, flat), slam.init(z, flat))
        last = z
        for cloud in (noisy, flat):
            p, err, nc = ctx.slam_localization_fast(cloud, pred + last, last)
            st = ctx.slam_fit_stats()
            _, corr, _, _ = slam.localize(cloud, pred + last, last)
            assert corr.shape[0] == 0 and nc == 0
            assert np.array_equal(st, np.zeros(5))
            check_fit(st, pred + last, last, p, err, nc)
            assert np.array_equal(ctx.slam_mapping(p, None), slam.map(p, cloud))
            last = p
    finally:
        ctx.close()
        slam.close()


def test_slam_run_single_frame_and_depth_input(pkg, oracle, synth):
    """nav_slam_run with one frame, and the depth-matrix input (prefetch_depth / depth_input=1) on a ragged
    shape: the same statistics and poses as the separate calls, checked against the oracle."""
    shape = (3, 257)
    r, c = shape
    n = 4
    depth = np.stack([synth.l5_depth_frame(f, r, c) for f in range(n)])
    clouds = np.stack([oracle.convert(d) for d in depth])
    step = np.array([-19.0, 0.3, 0.0, 0.0, 0.0, 0.0])
    z = np.zeros(6)
    slam = oracle.slam(r, c, 1)
    ctx = pkg.Context(r, c, device=0)
    with pinned(pkg, depth, clouds):
        try:
            # one frame
            ctx.slam_init(z, clouds[0], want_global=False)
            slam.init(z, clouds[0])
            poses, errs, ncs = ctx.slam_run([ptr(clouds[1])], step[None], z)
            st = ctx.slam_fit_stats()
            _, corr, _, _ = slam.localize(clouds[1], z + step, z)
            assert ncs[0] == corr.shape[0]
            check_stats(st, corr, shape)
            check_fit(st, z + step, z, poses[0], errs[0], ncs[0])
            assert np.array_equal(ctx.slam_mapping(poses[0], None), slam.map(poses[0], clouds[1]))
            # depth input through the separate calls
            ctx.slam_init(z, clouds[0], want_global=False)
            slam.init(z, clouds[0])
            got, last = [], z
            ctx.slam_prefetch(depth_ptr=ptr(depth[1]))
            for f in range(1, n):
                if f + 1 < n:
                    ctx.slam_prefetch(depth_ptr=ptr(depth[f + 1]))
                p, err, nc = ctx.slam_localization_fast_ptr(None, last + step, last)
                st = ctx.slam_fit_stats()
                _, corr, _, _ = slam.localize(clouds[f], last + step, last)
                assert nc == corr.shape[0]
                check_stats(st, corr, shape)
                check_fit(st, last + step, last, p, err, nc)
                assert np.array_equal(ctx.slam_mapping(p, None), slam.map(p, clouds[f]))
                got.append((p, err, nc, st))
                last = p
            # and as one nav_slam_run with depth_input = 1
            ctx.slam_init(z, clouds[0], want_global=False)
            poses, errs, ncs = ctx.slam_run([ptr(depth[f]) for f in range(1, n)], np.tile(step, (n - 1, 1)), z,
                                            depth_input=True)
            for f in range(n - 1):
                assert np.array_equal(poses[f], got[f][0]) and errs[f] == got[f][1] and ncs[f] == got[f][2]
            assert np.array_equal(ctx.slam_fit_stats(), got[-1][3])
        finally:
            ctx.close()
            slam.close()


# ------------------------------------------------------------------ entry points mixed on one context --------
@pytest.mark.parametrize("shape", [(16, 1800), (2, 4100)])
def test_closed_loop_mixed_with_other_entry_points(pkg, oracle, synth, shape):
    """One context, one map carried from call to call: nav_slam_run, the pipelined front end, the closed loop
    with and without prefetch, the blocking front end, and prefetches three ahead with the mapping deferred.
    Every output is compared bit for bit with the oracle driven along the same pose chain."""
    r, c = shape
    n = 22
    frames = np.stack([synth.room_frame(r, c, f) for f in range(n)])
    outs = {k: np.zeros((5,) + s, dtype=t) for k, s, t in (("feature_out", (r, c), np.int32),
                                                           ("nn_idx_out", (r, c), np.int32),
                                                           ("nn_dist_out", (r, c), np.float64),
                                                           ("global_out", (r, c, 3), np.float64))}
    z = np.zeros(6)
    fstep_pred = np.array([49.0, 1.0, 0.0, 0.0, 0.0, 0.2])
    fstep_final = np.array([50.0, 0.0, 0.0, 0.0, 0.0, 0.0])
    slam = oracle.slam(r, c, 1)
    ctx = pkg.Context(r, c, device=0)

    def oracle_loop_frame(f, pred, last, p, err, nc, st):
        _, corr, _, _ = slam.localize(frames[f], pred, last)
        assert nc == corr.shape[0]
        check_stats(st, corr, shape)
        check_fit(st, pred, last, p, err, nc)
        return slam.map(p, frames[f])

    def run(first, count, last):
        poses, errs, ncs = ctx.slam_run([ptr(frames[f]) for f in range(first, first + count)],
                                        np.tile(STEP, (count, 1)), last)
        st = ctx.slam_fit_stats()   # of the last frame
        for k in range(count):
            pred = last + STEP
            _, corr, _, _ = slam.localize(frames[first + k], pred, last)
            assert ncs[k] == corr.shape[0]
            if k == count - 1:
                check_stats(st, corr, shape)
                check_fit(st, pred, last, poses[k], errs[k], ncs[k])
            og = slam.map(poses[k], frames[first + k])
            last = poses[k]
        return last, og

    def submit(fs, last):
        chain = []
        for k, f in enumerate(fs):
            pred, final = last + fstep_pred, last + fstep_final
            ctx.frontend_submit(pred, last, final, cloud=ptr(frames[f]),
                                **{name: ptr(buf[k]) for name, buf in outs.items()})
            chain.append((f, pred, last, final))
            last = final
        return chain, last

    def check_submitted(chain):
        for k, (f, pred, last, final) in enumerate(chain):
            want = slam.frontend_frame(frames[f], pred, last, final)
            for name, w in zip(("feature_out", "nn_idx_out", "nn_dist_out", "global_out"), want):
                assert np.array_equal(outs[name][k], w), (f, name)

    with pinned(pkg, frames, *outs.values()):
        try:
            assert np.array_equal(ctx.slam_init(z, frames[0]), slam.init(z, frames[0]))
            # 1. nav_slam_run, then the pipelined front end (its streams and slots after the prefetch's)
            last, og = run(1, 3, z)
            chain, last = submit([4, 5, 6], last)
            ctx.frontend_wait()
            check_submitted(chain)
            # 2. two pipelined frames in flight, then the closed loop without prefetch
            chain, last = submit([7, 8], last)
            pred = last + STEP
            p, err, nc = ctx.slam_localization_fast(frames[9], pred, last)
            g = ctx.slam_mapping(p, None)
            ctx.frontend_wait()
            check_submitted(chain)
            assert np.array_equal(g, oracle_loop_frame(9, pred, last, p, err, nc, ctx.slam_fit_stats()))
            last = p
            # 3. closed loop with prefetch, the blocking front end, nav_slam_run again
            ctx.slam_prefetch(cloud_ptr=ptr(frames[10]))
            for f in (10, 11, 12):
                if f < 12:
                    ctx.slam_prefetch(cloud_ptr=ptr(frames[f + 1]))
                pred = last + STEP
                p, err, nc = ctx.slam_localization_fast_ptr(ptr(frames[f]), pred, last)
                g = ctx.slam_mapping(p, None)
                assert np.array_equal(g, oracle_loop_frame(f, pred, last, p, err, nc, ctx.slam_fit_stats()))
                last = p
            pred, final = last + fstep_pred, last + fstep_final
            a = ctx.frontend_frame(frames[13], pred, last, final)
            for x, y in zip(a, slam.frontend_frame(frames[13], pred, last, final)):
                assert np.array_equal(x, y)
            last, og = run(14, 3, final)
            assert np.array_equal(ctx.slam_mapping(last, None), og)   # the same pose again: the map comes back
            # 4. three prefetched ahead with the mapping deferred: the slot of the frame matched last stays
            # busy until nav_slam_mapping has queued its map
            ctx.slam_prefetch(cloud_ptr=ptr(frames[17]))
            ctx.slam_prefetch(cloud_ptr=ptr(frames[18]))
            pred = last + STEP
            p, err, nc = ctx.slam_localization_fast_ptr(None, pred, last)
            st = ctx.slam_fit_stats()
            ctx.slam_prefetch(cloud_ptr=ptr(frames[19]))
            with pytest.raises(pkg.NavError, match="nav_slam_mapping"):
                ctx.slam_prefetch(cloud_ptr=ptr(frames[20]))
            g = ctx.slam_mapping(p, None)
            assert np.array_equal(g, oracle_loop_frame(17, pred, last, p, err, nc, st))
            last = p
            ctx.slam_prefetch(cloud_ptr=ptr(frames[20]))   # now the slot is free
            for f in (18, 19, 20):
                pred = last + STEP
                p, err, nc = ctx.slam_localization_fast_ptr(None, pred, last)
                g = ctx.slam_mapping(p, None)
                assert np.array_equal(g, oracle_loop_frame(f, pred, last, p, err, nc, ctx.slam_fit_stats()))
                last = p
        finally:
            ctx.close()
            slam.close()
