"""The nearest-neighbour searches far from the origin and at extreme magnitudes, against the oracle bit for bit.

Two searches cull in reduced precision and stay exact only through a rounding argument: the per-row search of the
frame path (fp32 leaf and super boxes rounded outward, the query bracketed by a round-down and a round-up copy,
lower bounds formed with round-down arithmetic; k_frame_match, k_frame_seq, k_loop_step) and the tensor-core
brute force (bf16 splits accumulated in fp32, then an fp64 re-rank).  Near the origin one fp32 ulp is far below
the point spacing and no prune decision depends on a rounding direction.  Here the whole pose chain is moved by
an offset O, to where one fp32 ulp holds several points (1e6 .. 1.1e9 mm), where binary64 itself quantises the
points and makes organic distance ties (2^53, 1e17), and beyond FLT_MAX (1e39), where every row collapses to one
point and every query ties with every map point.  The large-map searches (kd tree with both split rules and all
three search kernels, the fp64 brute force, the tensor-core path) get point sets far from the origin, quantised
by binary64, stretched by outliers, queried from beyond FLT_MAX, and subnormal."""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from test_closed_loop_exact import check_fit, check_stats, loop_frames, pinned

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MIX = np.array([1.0, -0.75, 0.5])
# fp32 ulp at the offset 0.06 / 2 / 8 / 64-128 mm; binary64 ulp 1-2 / 16 mm; beyond FLT_MAX
OFFSETS = {"0": np.zeros(3), "1e6": 1e6 * MIX, "3e7": 3e7 * MIX, "1.2e8": 1.2e8 * MIX, "1.1e9": 1.1e9 * MIX,
           "x1.1e9": np.array([1.1e9, 0.0, 0.0]), "2^53": 2.0 ** 53 * MIX, "1e17": 1e17 * MIX, "1e39": 1e39 * MIX}
# the first three take the warp-cooperative culling (rows <= 2048 columns), the last two the super boxes
SHAPES = [(16, 1800), (64, 2048), (3, 257), (2, 4100), (1, 14000)]
MOTIONS = ["small", "large", "scrambled"]
STEP = {"small": np.array([46.0, 2.0, -1.0, 0.0, 0.0, 0.0]), "scrambled": np.array([46.0, 2.0, -1.0, 0.0, 0.0, 0.0]),
        "large": np.array([46.0, 2.0, -1.0, 0.0, 0.0, 30.0])}
PRED_OFF = np.array([3.0, -2.0, 1.0, 0.0, 0.0, 0.3])   # the prediction differs from the final pose


def pose0(offset):
    return np.concatenate([OFFSETS[offset], np.zeros(3)])


def pose_chain(p0, motion, n):
    """(pred, last, final) of frames 1 .. n-1: the queries of frame f use pred and last, its map final."""
    chain, last = [], p0
    for _ in range(1, n):
        final = last + STEP[motion]
        chain.append((final + PRED_OFF, last, final))
        last = final
    return chain


def assert_frame(got, want, ctx_msg):
    for name, x, y in zip(("labels", "nn_idx", "nn_dist", "global"), got, want):
        assert x.dtype == y.dtype and np.array_equal(x, y), (ctx_msg, name)


CASES = [(o, s, m) for o in OFFSETS for s in SHAPES for m in MOTIONS]
CASE_IDS = [f"{o}-{s[0]}x{s[1]}-{m}" for o, s, m in CASES]
SHAPE_IDS = [f"{r}x{c}" for r, c in SHAPES]


# ------------------------------------------------------------------ k_frame_match ------------------------------
@pytest.mark.parametrize("offset,shape,motion", CASES, ids=CASE_IDS)
def test_frontend_frame_far_from_origin(pkg, oracle, synth, offset, shape, motion):
    r, c = shape
    n = 3
    frames = loop_frames(synth, shape, motion, n)
    p0 = pose0(offset)
    ctx = pkg.Context(r, c, device=0)
    slam = oracle.slam(r, c, 1)
    try:
        assert np.array_equal(ctx.slam_init(p0, frames[0]), slam.init(p0, frames[0]))
        for f, (pred, last, final) in enumerate(pose_chain(p0, motion, n), start=1):
            want = slam.frontend_frame(frames[f], pred, last, final)
            assert (want[1] >= 0).sum() > 0
            assert_frame(ctx.frontend_frame(frames[f], pred, last, final), want, f)
    finally:
        ctx.close()
        slam.close()


# ------------------------------------------------------------------ k_frame_seq --------------------------------
@pytest.mark.parametrize("offset,shape,motion", CASES, ids=CASE_IDS)
def test_sequence_dev_far_from_origin(pkg, oracle, synth, offset, shape, motion):
    """nav_frontend_sequence_dev stopped after k frames leaves what the oracle has after k frames."""
    torch = pytest.importorskip("torch")
    from test_gpu_parity import _dev_to_numpy as dev_to_numpy
    r, c = shape
    n = 4
    frames = loop_frames(synth, shape, motion, n)
    p0 = pose0(offset)
    chain = pose_chain(p0, motion, n)
    pred, last, final = (np.stack([x[i] for x in chain]) for i in range(3))
    slam = oracle.slam(r, c, 1)
    slam.init(p0, frames[0])
    want = {f: slam.frontend_frame(frames[f], *chain[f - 1]) for f in range(1, n)}
    slam.close()
    d_frames = torch.from_numpy(frames).cuda()
    stream = torch.cuda.Stream()
    ctx = pkg.Context(r, c, device=0)
    try:
        ctx.set_stream(stream.cuda_stream)
        for k in (2, n - 1):
            ctx.slam_init_dev(d_frames[0].data_ptr(), p0)
            ctx.frontend_sequence_dev(d_frames[1].data_ptr(), k, pred[:k], last[:k], final[:k])
            stream.synchronize()
            res = ctx.frame_results_dev()
            got = (dev_to_numpy(torch, res.labels, np.int32, r * c).reshape(r, c),
                   dev_to_numpy(torch, res.nn_idx, np.int32, r * c).reshape(r, c),
                   dev_to_numpy(torch, res.nn_dist, np.float64, r * c).reshape(r, c),
                   dev_to_numpy(torch, res.global_, np.float64, r * c * 3).reshape(r, c, 3))
            ofeat, oidx, odist, og = want[k]
            lab = ofeat == 1
            assert np.array_equal(got[0], ofeat), k
            assert np.array_equal(got[1][lab], oidx[lab]) and np.array_equal(got[2][lab], odist[lab]), k
            assert np.array_equal(got[3], og), k
    finally:
        ctx.close()


# ------------------------------------------------------------------ two sequences, one of them far -------------
@pytest.mark.parametrize("shape", SHAPES, ids=SHAPE_IDS)
@pytest.mark.parametrize("motion", MOTIONS)
def test_two_sequences_one_far(pkg, oracle, synth, shape, motion):
    """n_seq = 2: sequence 0 at the origin, sequence 1 at 1.1e9 mm, in the same launches."""
    r, c = shape
    n = 3
    one = loop_frames(synth, shape, motion, n)
    frames = np.ascontiguousarray(np.stack([one, one], axis=1))   # the same frames at both offsets
    p0 = np.stack([pose0("0"), pose0("1.1e9")])
    ctx = pkg.Context(r, c, device=0, n_seq=2)
    slams = [oracle.slam(r, c, 1) for _ in range(2)]
    try:
        g = ctx.slam_init(p0, frames[0])
        for s in range(2):
            assert np.array_equal(g[s], slams[s].init(p0[s], frames[0, s]))
        chains = [pose_chain(p0[s], motion, n) for s in range(2)]
        for f in range(1, n):
            pred, last, final = (np.stack([chains[s][f - 1][i] for s in range(2)]) for i in range(3))
            got = ctx.frontend_frame(frames[f], pred, last, final)
            for s in range(2):
                assert_frame([x[s] for x in got], slams[s].frontend_frame(frames[f, s], pred[s], last[s], final[s]),
                             (f, s))
    finally:
        ctx.close()
        for sl in slams:
            sl.close()


# ------------------------------------------------------------------ the closed loop (k_loop_step) ---------------
@pytest.mark.parametrize("offset,shape,motion", CASES, ids=CASE_IDS)
def test_closed_loop_far_from_origin(pkg, oracle, synth, offset, shape, motion):
    """prefetch + nav_slam_localization_fast + nav_slam_mapping, then the same frames as one nav_slam_run.  At 2^53
    every global coordinate is a multiple of 1/2, every r a multiple of 1/2 and every |r|^2 a multiple of 1/4, all
    far below 2^50: the sums are exact in any order."""
    r, c = shape
    n = 4
    frames = loop_frames(synth, shape, motion, n)
    step = STEP[motion]
    p0 = pose0(offset)
    slam = oracle.slam(r, c, 1)
    ctx = pkg.Context(r, c, device=0)
    with pinned(pkg, frames):
        try:
            assert np.array_equal(ctx.slam_init(p0, frames[0]), slam.init(p0, frames[0]))
            got, last = [], p0
            ctx.slam_prefetch(cloud_ptr=frames[1].ctypes.data)
            for f in range(1, n):
                if f + 1 < n:
                    ctx.slam_prefetch(cloud_ptr=frames[f + 1].ctypes.data)
                pred = last + step
                p, err, nc = ctx.slam_localization_fast_ptr(frames[f].ctypes.data, pred, last)
                st = ctx.slam_fit_stats()
                _, corr, _, _ = slam.localize(frames[f], pred, last)
                assert nc == corr.shape[0] and nc > 0
                check_stats(st, corr, shape, exact=offset == "2^53")
                check_fit(st, pred, last, p, err, nc)
                assert np.array_equal(ctx.slam_mapping(p, None), slam.map(p, frames[f]))
                got.append((p, err, nc, st))
                last = p
            ctx.close()
            ctx = pkg.Context(r, c, device=0)
            ctx.slam_init(p0, frames[0], want_global=False)
            poses, errs, ncs = ctx.slam_run([frames[f].ctypes.data for f in range(1, n)], np.tile(step, (n - 1, 1)), p0)
            for f in range(n - 1):
                assert np.array_equal(poses[f], got[f][0]) and errs[f] == got[f][1] and ncs[f] == got[f][2]
            assert np.array_equal(ctx.slam_fit_stats(), got[-1][3])
        finally:
            ctx.close()
            slam.close()


# ------------------------------------------------------------------ a diverged pose -----------------------------
@pytest.mark.parametrize("shape", SHAPES, ids=SHAPE_IDS)
def test_diverged_pose_finds_no_match(pkg, oracle, synth, shape):
    """Frame 0 mapped at the origin, frame 1 localised with pred and last both moved by 1e160: every query sits near
    1e160 and its dsq to every map point overflows to +inf.  Every labelled pixel gets nn_idx = -1 and
    nn_dist = +inf, the closed loop finds no correspondence, and its pose is the fit with N = 0."""
    r, c = shape
    f0, f1 = loop_frames(synth, shape, "small", 2)
    z = np.zeros(6)
    last = np.concatenate([1e160 * MIX, np.zeros(3)])
    pred = last + STEP["small"]
    final = STEP["small"]
    slam = oracle.slam(r, c, 1)
    ctx = pkg.Context(r, c, device=0)
    try:
        # the front end
        assert np.array_equal(ctx.slam_init(z, f0), slam.init(z, f0))
        got = ctx.frontend_frame(f1, pred, last, final)
        want = slam.frontend_frame(f1, pred, last, final)
        assert_frame(got, want, "frontend")
        lab = got[0] == 1
        assert lab.sum() > 0
        assert np.all(got[1][lab] == -1) and np.all(got[2][lab] == np.inf)
        # the closed loop, separate calls and nav_slam_run
        slam.init(z, f0)
        ctx.slam_init(z, f0, want_global=False)
        p, err, nc = ctx.slam_localization_fast(f1, pred, last)
        st = ctx.slam_fit_stats()
        p_or, corr, _, _ = slam.localize(f1, pred, last)
        assert nc == 0 and corr.shape[0] == 0 and np.array_equal(st, np.zeros(5))
        check_fit(st, pred, last, p, err, nc)
        assert np.array_equal(p, p_or)
        assert np.array_equal(ctx.slam_mapping(p, None), slam.map(p, f1))
        with pinned(pkg, f1):
            ctx.slam_init(z, f0, want_global=False)
            poses, errs, ncs = ctx.slam_run([f1.ctypes.data], (pred - last)[None], last)
        assert ncs[0] == 0 and np.array_equal(ctx.slam_fit_stats(), np.zeros(5))
        check_fit(np.zeros(5), last + (pred - last), last, poses[0], errs[0], ncs[0])
    finally:
        ctx.close()
        slam.close()


# ------------------------------------------------------------------ large-map searches ---------------------------
NN_KINDS = ["far_dense", "quantised", "outliers", "outlier_1e20", "huge_queries", "subnormal"]
NN_SIZES = [1, 33, 4097, 70001]


def nn_set(kind, n):
    """(points, queries) of one family; nq = min(5000, 3 n + 64)."""
    rng = np.random.default_rng(NN_KINDS.index(kind) * 1000003 + n)
    nq = min(5000, 3 * n + 64)
    if kind == "far_dense":
        # a 10^4 mm cube centred at (1e9, -1e9, 5e8): a lattice with 1 mm jitter
        k = int(np.ceil(n ** (1 / 3)))
        g = np.stack(np.meshgrid(*[np.arange(k)] * 3, indexing="ij"), -1).reshape(-1, 3)[rng.permutation(k ** 3)[:n]]
        centre = np.array([1e9, -1e9, 5e8])
        pts = centre + (g + 0.5) * (1e4 / k) - 5e3 + rng.normal(0, 1, (n, 3))
        q = centre + rng.uniform(-5e3, 5e3, (nq, 3))
        q[: nq // 2] = pts[rng.integers(0, n, nq // 2)] + rng.normal(0, 0.5, (nq // 2, 3))
        q[:8] = pts[rng.integers(0, n, 8)]   # exact copies: dsq 0
    elif kind == "quantised":
        # binary64 ulp 1-2 mm at 2^53: duplicates and ties
        base = 2.0 ** 53 * MIX
        pts = base + rng.normal(0, 50, (n, 3))
        q = base + rng.normal(0, 50, (nq, 3))
    elif kind in ("outliers", "outlier_1e20"):
        # the bounding box stretched beyond what fp32 holds of |p - centre|^2 (and, with 1e39, of |p - centre|)
        pts = rng.normal(0, 100, (n, 3))
        far = [[1e20, 0.0, 0.0]] if kind == "outlier_1e20" else [[1e20, 0.0, 0.0], [0.0, -3e19, 0.0], [0.0, 0.0, 1e39]]
        for i, p in enumerate(far):
            pts[(i * 7919) % n] = p
        q = rng.normal(0, 100, (nq, 3))
    elif kind == "huge_queries":
        pts = rng.normal(0, 100, (n, 3))
        q = rng.normal(0, 100, (nq, 3))
        # beyond FLT_MAX; finite dsq 1e300; dsq overflowing (no answer); beyond what fp32 holds of q'.p'
        q[:4] = [[1e39, 0.0, 0.0], [1e150, 0.0, 0.0], [-1e300, 1e300, 0.0], [3e19, 0.0, 0.0]]
    else:   # subnormal: every dsq underflows to 0 -- exact ties everywhere
        pts = rng.normal(0, 1, (n, 3)) * 1e-310
        q = rng.normal(0, 1, (nq, 3)) * 1e-310
        pts[rng.random((n, 3)) < 0.2] = 0.0
        pts[rng.random((n, 3)) < 0.2] = -0.0
        q[rng.random((nq, 3)) < 0.2] = -0.0
    return np.ascontiguousarray(pts), np.ascontiguousarray(q)


NN_CASES = [(k, n) for k in NN_KINDS for n in NN_SIZES]


@pytest.fixture(scope="module")
def nn_answers(oracle):
    """oracle.nn_brute of every set, computed once."""
    out = {}
    for kind, n in NN_CASES:
        pts, q = nn_set(kind, n)
        out[kind, n] = (pts, q) + oracle.nn_brute(pts, q)
    return out


def assert_nn(idx, dist, oi, od, msg):
    assert np.array_equal(idx, oi), (msg, np.nonzero(idx != oi)[0][:8])
    assert np.array_equal(dist, od), (msg, np.nonzero(dist != od)[0][:8])


@pytest.mark.parametrize("kind,n", NN_CASES)
def test_large_map_searches(pkg, nn_answers, kind, n):
    """The kd tree (both split rules, host entry points and build_dev / nn_batch_dev on a user stream), the fp64
    brute force and the tensor-core path, each against oracle.nn_brute."""
    torch = pytest.importorskip("torch")
    pts, q, oi, od = nn_answers[kind, n]
    if kind == "huge_queries":
        assert oi[2] == -1 and od[2] == np.inf and oi[0] >= 0 and np.isfinite(od[1])
    nq = q.shape[0]
    for split in ("widest", "cyclic"):
        tree = pkg.KdTree(pts, device=0, split=split)
        try:
            idx, dist, near = tree.nn_batch(q)
        finally:
            tree.close()
        assert_nn(idx, dist, oi, od, ("host", split))
        assert np.array_equal(near[oi >= 0], pts[oi[oi >= 0]])
    stream = torch.cuda.Stream()
    sh = stream.cuda_stream
    with torch.cuda.stream(stream):   # every copy, fill and library call below on one user stream
        d_pts, d_q = torch.from_numpy(pts).cuda(), torch.from_numpy(q).cuda()
        d_idx = torch.empty(nq, dtype=torch.int32, device="cuda")
        d_dist = torch.empty(nq, dtype=torch.float64, device="cuda")
        for split in ("widest", "cyclic"):
            tree = pkg.KdTree(dev_ptr=d_pts.data_ptr(), n=n, stream=sh, split=split)
            try:
                d_idx.fill_(7)
                d_dist.fill_(7.0)
                tree.nn_batch_dev(d_q.data_ptr(), nq, d_idx.data_ptr(), d_dist.data_ptr(), stream=sh)
                assert_nn(d_idx.cpu().numpy(), d_dist.cpu().numpy(), oi, od, ("dev", split))
            finally:
                tree.close()
        for tc in (False, True):
            d_idx.fill_(7)
            d_dist.fill_(7.0)
            pkg.bruteforce_nn_dev(0, d_pts.data_ptr(), n, d_q.data_ptr(), nq, d_idx.data_ptr(), d_dist.data_ptr(),
                                  use_tensor_cores=tc, stream=sh)
            assert_nn(d_idx.cpu().numpy(), d_dist.cpu().numpy(), oi, od, "tensor cores" if tc else "fp64 brute force")


# ------------------------------------------------------------------ the stackless kd kernels -------------------
BIG_N, BIG_NQ = 70001, 262144   # > 12 * 148 * 128 queries: every lane of k_kd_nn_conv refills more than once


def big_case():
    pts, _ = nn_set("far_dense", BIG_N)
    rng = np.random.default_rng(5)
    q = pts[rng.integers(0, BIG_N, BIG_NQ)] + rng.normal(0, 30, (BIG_NQ, 3))
    return pts, np.ascontiguousarray(q)


@pytest.mark.parametrize("kernel", ["plain", "conv"])
def test_stackless_kd_kernels(pkg, oracle, nn_answers, kernel):
    """NAV_KD_KERNEL=plain|conv (k_kd_nn, k_kd_nn_conv) is read once per process, so a worker process answers every
    set of test_large_map_searches with both split rules, plus 262 144 queries on a 70 001-point map; the big case
    is held to the default kernel and the fp64 brute force, and to the oracle on 2000 queries."""
    torch = pytest.importorskip("torch")
    bp, bq = big_case()
    with tempfile.TemporaryDirectory() as tmp:
        src, dst = os.path.join(tmp, "in.npz"), os.path.join(tmp, "out.npz")
        arrays = {"big_pts": bp, "big_q": bq}
        for i, (kind, n) in enumerate(NN_CASES):
            arrays[f"pts_{i}"], arrays[f"q_{i}"] = nn_answers[kind, n][:2]
        np.savez(src, n_cases=len(NN_CASES), **arrays)
        res = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "kd_kernel_worker.py"), src, dst],
                             env=dict(os.environ, NAV_KD_KERNEL=kernel), capture_output=True, text=True, timeout=900)
        assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
        got = dict(np.load(dst))
    for i, (kind, n) in enumerate(NN_CASES):
        _, _, oi, od = nn_answers[kind, n]
        for split in ("widest", "cyclic"):
            assert_nn(got[f"idx_{i}_{split}"], got[f"dist_{i}_{split}"], oi, od, (kernel, kind, n, split))
    tree = pkg.KdTree(bp, device=0)
    try:
        ki, kd, _ = tree.nn_batch(bq)
    finally:
        tree.close()
    d_pts, d_q = torch.from_numpy(bp).cuda(), torch.from_numpy(bq).cuda()
    d_idx = torch.empty(BIG_NQ, dtype=torch.int32, device="cuda")
    d_dist = torch.empty(BIG_NQ, dtype=torch.float64, device="cuda")
    pkg.bruteforce_nn_dev(0, d_pts.data_ptr(), BIG_N, d_q.data_ptr(), BIG_NQ, d_idx.data_ptr(), d_dist.data_ptr(),
                          stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    bi, bd = d_idx.cpu().numpy(), d_dist.cpu().numpy()
    for split in ("widest", "cyclic"):
        gi, gd = got[f"big_idx_{split}"], got[f"big_dist_{split}"]
        assert_nn(gi, gd, ki, kd, (kernel, "big vs default kernel", split))
        assert_nn(gi, gd, bi, bd, (kernel, "big vs fp64 brute force", split))
        oi, od = oracle.nn_brute(bp, bq[:2000])
        assert_nn(gi[:2000], gd[:2000], oi, od, (kernel, "big vs oracle", split))
