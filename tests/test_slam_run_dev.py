"""nav_slam_run_dev: the closed loop of nav_slam_run on device-resident frames, with the pose fit on the GPU, for one
or many sequences in the same launches.

Every output is held bit for bit to nav_slam_run on pinned host copies of the same frames (poses, RMS errors,
correspondence counts) and to nav_slam_fit_stats after each of its frames (the totals); several sequences to
single-sequence replays; the context afterwards to the state nav_slam_run leaves, so that the host-driven calls
continue the trajectory.  The device fit itself goes through a test seam against the host fit and its restatement
in Python, including the branches frames cannot reach."""
import ctypes as C
import math

import numpy as np
import pytest

from test_closed_loop_exact import _C1, _C2, fit_py, pinned, ptr
from test_sequence_outputs import assert_same_state, ctx_state

gpu = pytest.mark.gpu
STEP = np.array([46.0, 2.0, -1.0, 0.0, 0.0, 0.0])


# ------------------------------------------------------------------ helpers ----------------------------------
def frames_of(synth, shape, n, n_seq=1, integer_mm=False, scrambled=False):
    """[n][n_seq][rows][cols][3] room frames (frame 0 is the one the map is initialised with)."""
    r, c = shape
    fr = np.stack([np.stack([synth.room_frame(r, c, f, seq=s, integer_mm=integer_mm) for s in range(n_seq)])
                   for f in range(n)])
    if scrambled:   # matches land in arbitrary tiles of the row
        rng = np.random.default_rng(r * 7919 + c)
        for f in range(n):
            for s in range(n_seq):
                fr[f, s] = fr[f, s][:, rng.permutation(c)]
    return np.ascontiguousarray(fr)


def deltas_of(k, n_seq, seed, rotate=True):
    """[k][n_seq][6] dead-reckoning increments, different per frame and sequence."""
    rng = np.random.default_rng(seed)
    d = np.tile(STEP, (k, n_seq, 1)) + rng.uniform(-3.0, 3.0, (k, n_seq, 6)) * np.array([1, 1, 1, 0, 0, 0])
    if rotate:
        d[..., 5] += rng.uniform(-0.4, 0.4, (k, n_seq))
        d[..., 3] += rng.uniform(-0.05, 0.05, (k, n_seq))
    return d


def host_loop(pkg, shape, frames1, deltas1, start, stepwise=True):
    """nav_slam_run on a single-sequence context mapped at `start` with frames1[0]; frames1[1:] are the loop.
    stepwise: one call per frame, which continues the trajectory, with nav_slam_fit_stats after each.
    Returns (ctx, poses [k,6], errors [k], n_corr [k], stats [k,5] or None)."""
    r, c = shape
    k = frames1.shape[0] - 1
    ctx = pkg.Context(r, c, device=0)
    ctx.slam_init(start, frames1[0], want_global=False)
    if not stepwise:
        poses, errs, ncs = ctx.slam_run([ptr(frames1[f]) for f in range(1, k + 1)], deltas1, start)
        return ctx, poses, errs, ncs, None
    poses, errs, ncs, stats = [], [], [], []
    last = np.asarray(start, dtype=np.float64)
    for f in range(k):
        p, e, n = ctx.slam_run([ptr(frames1[f + 1])], deltas1[f:f + 1], last)
        poses.append(p[0])
        errs.append(e[0])
        ncs.append(n[0])
        stats.append(ctx.slam_fit_stats())
        last = p[0]
    return ctx, np.array(poses), np.array(errs), np.array(ncs), np.array(stats)


class DevOut:
    """The three output buffers of nav_slam_run_dev on the device."""

    def __init__(self, torch, k, n_seq):
        self.poses = torch.full((k, n_seq, 6), -7.0, dtype=torch.float64, device="cuda")
        self.error = torch.full((k, n_seq), -7.0, dtype=torch.float64, device="cuda")
        self.stats = torch.full((k, n_seq, 5), -7.0, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()

    def ptrs(self):
        return self.poses.data_ptr(), self.error.data_ptr(), self.stats.data_ptr()

    def get(self):
        return self.poses.cpu().numpy(), self.error.cpu().numpy(), self.stats.cpu().numpy()


def dev_loop(pkg, torch, shape, frames, deltas, start):
    """nav_slam_run_dev on a fresh context of n_seq = frames.shape[1] mapped at start with frames[0]."""
    r, c = shape
    k, n_seq = frames.shape[0] - 1, frames.shape[1]
    ctx = pkg.Context(r, c, device=0, n_seq=n_seq)
    ctx.slam_init(start.reshape(n_seq, 6), frames[0] if n_seq > 1 else frames[0, 0], want_global=False)
    d_frames = torch.from_numpy(frames).cuda()
    out = DevOut(torch, k, n_seq)
    n0 = ctx.launch_count()
    ctx.slam_run_dev(d_frames[1].data_ptr(), k, deltas.reshape(-1, 6), start.reshape(n_seq, 6), *out.ptrs())
    ctx.synchronize()
    assert ctx.launch_count() - n0 == k + 1
    return ctx, out.get()


def same_bits(a, b):
    return np.ascontiguousarray(a, dtype=np.float64).tobytes() == np.ascontiguousarray(b, dtype=np.float64).tobytes()


def same_values(a, b):
    """same_bits, except that a NaN matches any NaN: its payload and sign follow the processor that formed it (the
    host's SSE units and the GPU give different NaN bits for the same invalid operation)."""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.dtype.kind != "f":
        return a.tobytes() == b.tobytes()
    na, nb = np.isnan(a), np.isnan(b)
    return bool((na == nb).all()) and a[~na].tobytes() == b[~nb].tobytes()


def loop_state(pkg, ctx):
    """What the closed loop leaves in the context: the last frame's nn_idx / nn_dist, the map (global cloud, masks)."""
    st = ctx_state(pkg, ctx, rows_to_export=(0, ctx.rows - 1))
    del st["labels"]   # nav_slam_run keeps the labels of its frames in the prefetch slots
    return st


# ------------------------------------------------------------------ 1. parity with the host loop -------------
PARITY = [((64, 2048), 40, False, False), ((5, 33), 6, False, False), ((3, 257), 6, False, True),
          ((2, 2048), 6, False, True), ((16, 1800), 8, False, False), ((2, 600), 5, False, True),
          ((3, 256), 5, True, False), ((16, 1800), 6, True, False),
          # the remaining cluster widths, 4 to 7 tiles
          ((2, 1000), 5, False, True), ((2, 1100), 5, False, True), ((2, 1500), 5, False, True),
          ((2, 1700), 5, False, True)]


@gpu
@pytest.mark.parametrize("shape,k,integer_mm,scrambled", PARITY)
def test_parity_with_host_loop(pkg, synth, shape, k, integer_mm, scrambled):
    """n_seq = 1: poses, errors and totals bit for bit those of nav_slam_run (one call per frame and one call for
    the whole loop), N = its n_corr_out; the context afterwards as nav_slam_run leaves it.  Integer-mm data with
    integer steps and no rotation: every sum is exact."""
    torch = pytest.importorskip("torch")
    frames = frames_of(synth, shape, k + 1, integer_mm=integer_mm, scrambled=scrambled)
    deltas = deltas_of(k, 1, seed=k * 31 + shape[1], rotate=not integer_mm)
    if integer_mm:
        deltas = np.rint(deltas)
    start = np.zeros(6)
    frames1 = np.ascontiguousarray(frames[:, 0])
    ctx, (poses, errs, stats) = dev_loop(pkg, torch, shape, frames, deltas, start)
    with pinned(pkg, frames1):
        hctx, hp, he, hn, hs = host_loop(pkg, shape, frames1, deltas[:, 0], start)
        hctx.close()
        hctx, hp1, he1, hn1, _ = host_loop(pkg, shape, frames1, deltas[:, 0], start, stepwise=False)
    try:
        assert same_bits(hp1, hp) and same_bits(he1, he) and np.array_equal(hn1, hn)
        assert same_bits(poses[:, 0], hp), poses[:, 0] - hp
        assert same_bits(errs[:, 0], he)
        assert same_bits(stats[:, 0], hs)
        assert np.array_equal(stats[:, 0, 0].astype(np.int64), hn)
        assert hn.sum() > 0
        for f in range(k):   # the device fit is the host fit
            last = start if f == 0 else hp[f - 1]
            want, want_err, want_n = fit_py(hs[f], last + deltas[f, 0], last)
            assert same_bits(want, hp[f]) and want_err == he[f] and want_n == hn[f]
        assert_same_state(loop_state(pkg, ctx), loop_state(pkg, hctx))
    finally:
        ctx.close()
        hctx.close()


# ------------------------------------------------------------------ 2. degenerate frames ----------------------
@gpu
def test_degenerate_frames(pkg, synth):
    """A frame with no labelled point, a blank previous frame (N = 0: the pose stays at the prediction, error 0),
    and a diverged increment that drives the distances to inf / NaN: the same bits as nav_slam_run."""
    torch = pytest.importorskip("torch")
    shape = (5, 33)
    r, c = shape
    rng = np.random.default_rng(5)
    flat = np.zeros((r, c, 3))
    flat[..., 0] = 1000.0   # all points identical: no labels
    room = [synth.room_frame(r, c, f) for f in range(8)]
    noisy = rng.normal(0, 1000, size=(r, c, 3))
    seq = [room[0], room[1], flat, room[2], noisy, flat, flat, room[3], room[4], room[5], room[6], room[7]]
    frames = np.ascontiguousarray(np.stack(seq)[:, None])
    k = frames.shape[0] - 1
    deltas = deltas_of(k, 1, seed=9)
    deltas[8, 0, 0] = 1e308      # the prediction overflows to inf: inf / NaN distances from here on
    deltas[9, 0, 0] = 1e308
    start = np.array([3.0, -2.0, 1.0, 0.5, 0.0, 2.0])
    ctx, (poses, errs, stats) = dev_loop(pkg, torch, shape, frames, deltas, start)
    frames1 = np.ascontiguousarray(frames[:, 0])
    with pinned(pkg, frames1):
        hctx, hp, he, hn, hs = host_loop(pkg, shape, frames1, deltas[:, 0], start)
    try:
        assert same_values(poses[:, 0], hp) and same_values(errs[:, 0], he) and same_values(stats[:, 0], hs)
        assert np.array_equal(stats[:, 0, 0].astype(np.int64), hn)
        assert same_bits(poses[:8, 0], hp[:8]) and same_bits(errs[:8, 0], he[:8])
        for f in (1, 2, 4, 5):   # no labels in the frame or in the map it is matched against
            assert hn[f] == 0 and he[f] == 0.0 and same_bits(hs[f], np.zeros(5))
            last = hp[f - 1]
            assert same_bits(hp[f], last + ((last + deltas[f, 0]) - last))
        assert not np.isfinite(hp[8:, 0]).any()
        a, b = loop_state(pkg, ctx), loop_state(pkg, hctx)
        assert a.keys() == b.keys()
        for key in a:
            for x, y in (zip(a[key], b[key]) if isinstance(a[key], tuple) else [(a[key], b[key])]):
                assert same_values(x, y), key
    finally:
        ctx.close()
        hctx.close()


# ------------------------------------------------------------------ 3. many sequences ------------------------
@gpu
@pytest.mark.parametrize("shape,n_seq,k", [((16, 1800), 3, 6), ((8, 600), 16, 5)])
def test_many_sequences(pkg, synth, shape, n_seq, k):
    """n_seq sequences with different starts and increments in the same launches: sequence s equals a
    single-sequence nav_slam_run_dev of it and nav_slam_run of it, bit for bit."""
    torch = pytest.importorskip("torch")
    frames = frames_of(synth, shape, k + 1, n_seq=n_seq)
    deltas = deltas_of(k, n_seq, seed=n_seq)
    start = np.array([[0.0, 0.5 * s, 0.0, 0.0, 0.0, 0.1 * s] for s in range(n_seq)])
    ctx, (poses, errs, stats) = dev_loop(pkg, torch, shape, frames, deltas, start)
    ctx.close()
    for s in range(n_seq):
        one = np.ascontiguousarray(frames[:, s:s + 1])
        c1, (p1, e1, s1) = dev_loop(pkg, torch, shape, one, np.ascontiguousarray(deltas[:, s:s + 1]), start[s])
        c1.close()
        assert same_bits(poses[:, s], p1[:, 0]) and same_bits(errs[:, s], e1[:, 0]) and same_bits(stats[:, s], s1[:, 0])
        frames1 = np.ascontiguousarray(frames[:, s])
        with pinned(pkg, frames1):
            hctx, hp, he, hn, hs = host_loop(pkg, shape, frames1, deltas[:, s], start[s])
            hctx.close()
        assert same_bits(poses[:, s], hp) and same_bits(errs[:, s], he) and same_bits(stats[:, s], hs), s


# ------------------------------------------------------------------ 4. continuation, mixed use ---------------
@gpu
def test_continuation_and_mixed_use(pkg, synth):
    """nav_slam_run_dev over frames [1, K], then nav_slam_run over [K+1, 2K] from the device's last pose: one
    nav_slam_run over [1, 2K].  The context then still serves nav_slam_localization_fast, nav_slam_mapping and the
    pipelined nav_frontend_submit, with the same results as the host-only context."""
    torch = pytest.importorskip("torch")
    shape = (16, 1800)
    r, c = shape
    K = 5
    frames = frames_of(synth, shape, 2 * K + 4)
    frames1 = np.ascontiguousarray(frames[:, 0])
    deltas = deltas_of(2 * K, 1, seed=77)
    z = np.zeros(6)
    outs = {k: np.zeros((2,) + s, dtype=t) for k, s, t in (("feature_out", (r, c), np.int32),
                                                           ("nn_idx_out", (r, c), np.int32),
                                                           ("nn_dist_out", (r, c), np.float64),
                                                           ("global_out", (r, c, 3), np.float64))}
    outs_h = {k: np.zeros_like(v) for k, v in outs.items()}
    ctx, (poses, errs, stats) = dev_loop(pkg, torch, shape, frames[:K + 1], deltas[:K], z)
    hctx = pkg.Context(r, c, device=0)
    with pinned(pkg, frames1, *outs.values(), *outs_h.values()):
        try:
            hctx.slam_init(z, frames1[0], want_global=False)
            hp, he, hn = hctx.slam_run([ptr(frames1[f]) for f in range(1, 2 * K + 1)], deltas[:, 0], z)
            assert same_bits(poses[:, 0], hp[:K]) and same_bits(errs[:, 0], he[:K])
            last = poses[K - 1, 0]
            p2, e2, n2 = ctx.slam_run([ptr(frames1[f]) for f in range(K + 1, 2 * K + 1)], deltas[K:, 0], last)
            assert same_bits(p2, hp[K:]) and same_bits(e2, he[K:]) and np.array_equal(n2, hn[K:])
            assert same_bits(ctx.slam_fit_stats(), hctx.slam_fit_stats())
            # the closed loop without prefetch, then the mapping
            last = hp[-1]
            pred = last + STEP
            a = ctx.slam_localization_fast(frames1[2 * K + 1], pred, last)
            b = hctx.slam_localization_fast(frames1[2 * K + 1], pred, last)
            assert same_bits(a[0], b[0]) and a[1] == b[1] and a[2] == b[2]
            assert same_bits(ctx.slam_mapping(a[0], None), hctx.slam_mapping(b[0], None))
            # the pipelined front end on both contexts
            last = a[0]
            for x, o in ((ctx, outs), (hctx, outs_h)):
                ll = last
                for j, f in enumerate((2 * K + 2, 2 * K + 3)):
                    x.frontend_submit(ll + STEP, ll, ll + STEP, cloud=ptr(frames1[f]),
                                      **{name: ptr(buf[j]) for name, buf in o.items()})
                    ll = ll + STEP
                x.frontend_wait()
            for name in outs:
                assert outs[name].tobytes() == outs_h[name].tobytes(), name
            # and the device loop once more, from where the pipelined frames left the map
            ll = last + 2 * STEP
            more = np.ascontiguousarray(frames[2 * K + 1:2 * K + 4])
            d_more = torch.from_numpy(more).cuda()
            o1, o2 = DevOut(torch, 2, 1), DevOut(torch, 2, 1)
            for x, o in ((ctx, o1), (hctx, o2)):
                x.slam_run_dev(d_more[1].data_ptr(), 2, deltas[:2, 0], ll, *o.ptrs())
                x.synchronize()
            for u, v in zip(o1.get(), o2.get()):
                assert same_bits(u, v)
        finally:
            ctx.close()
            hctx.close()


# ------------------------------------------------------------------ 5. the device fit -----------------------
DBL_MIN = 2.2250738585072014e-308


def fit_trace(st, pred, last):
    """fit_py's loop again, reporting what it went through: (iterations run before the tol break, or 200; whether
    some v[j] or vh was subnormal, i.e. 0 < |x| < DBL_MIN -- the operands that take the device's division and square
    root to their slow paths)."""
    lr, tol, b1, b2, eps = 0.1, 1e-6, 0.9, 0.999, 1e-8
    N, S, Q = float(st[0]), [float(x) for x in st[1:4]], float(st[4])
    t = [float(pred[k]) - float(last[k]) for k in range(3)]
    m, v = [0.0] * 3, [0.0] * 3
    prev = 0.0
    sub = False
    for it in range(200):
        total = Q - 2.0 * (t[0] * S[0] + t[1] * S[1] + t[2] * S[2]) + N * (t[0] * t[0] + t[1] * t[1] + t[2] * t[2])
        if N == 0:
            total = 0.0
        if abs(total - prev) < tol:
            return it, sub
        prev = total
        for j in range(3):
            g = -(S[j] - N * t[j]) / N if N > 0 else 0.0
            m[j] = b1 * m[j] + (1 - b1) * g
            v[j] = b2 * v[j] + (1 - b2) * g * g
            vh = v[j] / _C2[it]
            sub = sub or 0 < abs(v[j]) < DBL_MIN or 0 < abs(vh) < DBL_MIN
            t[j] -= lr * (m[j] / _C1[it]) / (math.sqrt(vh) + eps)
    return 200, sub


def fit_vectors(n, seed):
    """Random stat vectors, then (in the first rows) the edge cases, by name: N = 0, the tol break at the first
    iteration and after many, huge Q, overflow, subnormal v and vh, inf / NaN, a diverged prediction."""
    rng = np.random.default_rng(seed)
    N = rng.integers(1, 40000, n).astype(np.float64)
    S = rng.normal(0, 1, (n, 3)) * N[:, None] * rng.choice([1e-3, 1.0, 30.0, 1e4], (n, 1))
    Q = (S ** 2).sum(1) / N * rng.uniform(1.0, 5.0, n) + rng.uniform(0, 1e6, n)
    st = np.column_stack([N, S, Q])
    pred = rng.normal(0, 1, (n, 6)) * rng.choice([1.0, 100.0, 1e5], (n, 1))
    last = pred - rng.normal(0, 1, (n, 6)) * rng.choice([0.0, 1e-3, 1.0, 60.0], (n, 1))
    z6 = np.zeros(6)
    edge = {
        "n0": ([0, 0, 0, 0, 0], z6, z6),
        "n0_sums": ([0, 5.0, -3.0, 1.0, 7.0], np.arange(6.0), z6),   # the pose stays at the prediction
        "tol_first": ([10, 0, 0, 0, 0], z6, z6),                     # total stays 0: break at iteration 0
        "tol_late_a": ([10, 2e-3, 0, 0, 1.0], z6, z6),               # converges: break after dozens of iterations
        "tol_late_b": ([1, 0.0, 0, 0, 3e-6], np.array([1e-3, 0, 0, 0, 0, 0]), z6),
        "huge_q": ([3, 1.0, 2.0, 3.0, 1e300], z6, z6),
        "overflow": ([1e6, 1e300, -1e300, 1e300, 1e308], np.ones(6), z6),
        # |g| around 1e-158: g*g, v and vh subnormal, fed to sqrt and the division
        "sub_v": ([1, 1e-158, 0, 0, 1.0], z6, z6),
        "sub_v_3": ([1, 1e-157, -3e-159, 2e-160, 1.0], z6, z6),
        # the same in one component while another keeps the loop running for over a hundred iterations
        "sub_v_long": ([1, 1e-159, 5.0, -2e-160, 30.0], z6, z6),
        "sub_v_long_b": ([3, 4e-158, 12.0, 0, 80.0], z6, z6),
        "inf_s": ([7, np.inf, 1.0, 2.0, 3.0], z6, z6),
        "nan_s": ([7, np.nan, 1.0, 2.0, 3.0], z6, z6),
        "neg_q": ([7, 1.0, 2.0, 3.0, -5.0], z6, z6),                  # error from fmax(total, 0)
        "inf_pred": ([1, 0, 0, 0, 0], np.array([np.inf, 0, 0, 0, 0, 0]), z6),
        "nan_pred": ([1, 0, 0, 0, 0], np.array([np.nan, 0, 0, 1, 2, 3]), z6),
        "huge_t": ([5, 2.0, 2.0, 2.0, 9.0], np.array([1e308, -1e308, 0, 0, 0, 0]), np.array([-1e308, 1e308, 0, 0, 0, 0])),
    }
    idx = {}
    for i, (name, (s_, p_, q_)) in enumerate(edge.items()):
        st[i], pred[i], last[i] = s_, p_, q_
        idx[name] = i
    return st, pred, last, idx


def test_fit_edge_vectors_reach_their_branches():
    """The edge vectors of the device-fit test go where their names say (a CPU replay of the loop)."""
    st, pred, last, idx = fit_vectors(64, seed=11)
    trace = {k: fit_trace(st[i], pred[i], last[i]) for k, i in idx.items()}
    assert trace["tol_first"][0] == 0 and trace["n0"][0] == 0
    for k in ("tol_late_a", "tol_late_b"):
        assert 20 < trace[k][0] < 200, (k, trace[k])
    for k in ("sub_v", "sub_v_3", "sub_v_long", "sub_v_long_b"):
        assert trace[k][1] and trace[k][0] >= 1, (k, trace[k])
    for k in ("sub_v_long", "sub_v_long_b"):
        assert trace[k][0] > 100, (k, trace[k])


@gpu
def test_device_fit_matches_host_fit(pkg):
    """nav_debug_fit_from_stats_dev (the device fit_translation, tables uploaded from the host's pow()) on 10^5 stat
    vectors: bit for bit nav_slam_fit_from_stats on each (NaN for NaN), and fit_py on the edge cases and a sample."""
    torch = pytest.importorskip("torch")
    L = pkg.load_library()
    L.nav_debug_fit_from_stats_dev.argtypes = [C.c_void_p] * 3 + [C.c_size_t] + [C.c_void_p] * 3
    n = 100000
    st, pred, last, idx = fit_vectors(n, seed=11)
    n_edge = len(idx)
    d_st = torch.from_numpy(st).cuda()
    d_pred = torch.from_numpy(pred).cuda()
    d_last = torch.from_numpy(last).cuda()
    d_pose = torch.full((n, 6), -7.0, dtype=torch.float64, device="cuda")
    d_err = torch.full((n,), -7.0, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    assert L.nav_debug_fit_from_stats_dev(d_st.data_ptr(), d_pred.data_ptr(), d_last.data_ptr(), n, d_pose.data_ptr(),
                                          d_err.data_ptr(), None) == 0, L.nav_last_error()
    torch.cuda.synchronize()
    pose, err = d_pose.cpu().numpy(), d_err.cpu().numpy()
    bad = []
    for i in range(n):
        hp, he = pkg.fit_from_stats(st[i], pred[i], last[i])
        if not (same_values(hp, pose[i]) and same_values(he, err[i])):
            bad.append(i)
    assert not bad, (len(bad), bad[:10])
    rng = np.random.default_rng(12)
    for i in list(range(n_edge)) + list(rng.choice(np.arange(n_edge, n), 500, replace=False)):
        want, want_err, _ = fit_py(st[i], pred[i], last[i])
        if math.isnan(want_err):   # Python's max() keeps a NaN total where C's fmax() drops it: host fit above only
            continue
        assert same_values(want, pose[i]) and same_values(want_err, err[i]), i
    # the rare branches were taken
    i0, i1, inan = idx["n0"], idx["n0_sums"], idx["nan_s"]
    assert err[i0] == 0.0 and same_bits(pose[i1], last[i1] + (pred[i1] - last[i1]))
    assert math.isnan(err[inan]) or math.isnan(pose[inan][0])


# ------------------------------------------------------------------ 6. refusals, launch count ----------------
@gpu
def test_refusals_leave_the_context_unchanged(pkg, synth):
    """Every refusal returns an error naming the cause, queues nothing (nav_launch_count) and leaves the context
    as it was; n_frames = 0 returns 0 and writes nothing; a successful call adds n_frames + 1 launches."""
    torch = pytest.importorskip("torch")
    L = pkg.load_library()
    shape = (5, 33)
    r, c = shape
    k = 3
    frames = frames_of(synth, shape, k + 1)
    d_frames = torch.from_numpy(frames).cuda()
    deltas = deltas_of(k, 1, seed=3)
    z = np.zeros(6)
    host = np.zeros((k, 8))
    out = DevOut(torch, k, 1)
    pp, pe, ps = out.ptrs()

    fresh = pkg.Context(r, c, device=0)   # no map yet
    try:
        with pytest.raises(pkg.NavError, match="nav_slam_init"):
            fresh.slam_run_dev(d_frames[1].data_ptr(), k, deltas, z, pp, pe, ps)
        assert fresh.launch_count() == 0
    finally:
        fresh.close()
    wide = pkg.Context(2, 2049, device=0)
    try:
        wide.slam_init(z, synth.room_frame(2, 2049, 0), want_global=False)
        n0 = wide.launch_count()
        with pytest.raises(pkg.NavError, match="2048"):
            wide.slam_run_dev(d_frames[1].data_ptr(), 1, deltas[:1], z, pp, pe, ps)
        assert wide.launch_count() == n0
    finally:
        wide.close()

    ctx = pkg.Context(r, c, device=0)
    try:
        ctx.slam_init(z, frames[0, 0], want_global=False)
        before = ctx_state(pkg, ctx)
        n0 = ctx.launch_count()
        dp = (pkg.binding.NavPos * k)(*[pkg.binding.NavPos(*row) for row in deltas.reshape(k, 6)])
        start = pkg.binding.NavPos(*z)
        good = pkg.binding.NavRunDevOut(pp, pe, ps)
        raw = L.nav_slam_run_dev
        cases = [
            (lambda: raw(ctx.h, d_frames[1].data_ptr(), k, dp, C.byref(start), None), "null"),
            (lambda: raw(ctx.h, d_frames[1].data_ptr(), k, dp, C.byref(start),
                         C.byref(pkg.binding.NavRunDevOut(None, pe, ps))), "null"),
            (lambda: raw(ctx.h, d_frames[1].data_ptr(), k, None, C.byref(start), C.byref(good)), "null"),
            (lambda: raw(ctx.h, d_frames[1].data_ptr(), k, dp, None, C.byref(good)), "null"),
            (lambda: raw(ctx.h, None, k, dp, C.byref(start), C.byref(good)), "null"),
            (lambda: raw(ctx.h, d_frames[1].data_ptr(), -1, dp, C.byref(start), C.byref(good)), "negative"),
            (lambda: raw(ctx.h, host.ctypes.data, k, dp, C.byref(start), C.byref(good)), "dev_frames"),
            (lambda: raw(ctx.h, d_frames[1].data_ptr(), k, dp, C.byref(start),
                         C.byref(pkg.binding.NavRunDevOut(host.ctypes.data, pe, ps))), "out->poses"),
            (lambda: raw(ctx.h, d_frames[1].data_ptr(), k, dp, C.byref(start),
                         C.byref(pkg.binding.NavRunDevOut(pp, host.ctypes.data, ps))), "out->error"),
            (lambda: raw(ctx.h, d_frames[1].data_ptr(), k, dp, C.byref(start),
                         C.byref(pkg.binding.NavRunDevOut(pp, pe, host.ctypes.data))), "out->fit_stats"),
        ]
        for call, word in cases:
            assert call() != 0
            assert word in L.nav_last_error().decode(), (word, L.nav_last_error())
            assert ctx.launch_count() == n0
        ctx.set_tie_rule("reference")
        with pytest.raises(pkg.NavError, match="NAV_TIE_REFERENCE"):
            ctx.slam_run_dev(d_frames[1].data_ptr(), k, deltas, z, pp, pe, ps)
        ctx.set_tie_rule("lowest_index")
        assert ctx.launch_count() == n0
        # n_frames = 0: success, nothing queued, nothing written
        ctx.slam_run_dev(d_frames[1].data_ptr(), 0, np.zeros((0, 6)), z, pp, pe, ps)
        assert ctx.launch_count() == n0
        assert all((a == -7.0).all() for a in out.get())
        assert_same_state(before, ctx_state(pkg, ctx))
        # a call that runs: n_frames + 1 launches (ctx_state itself launches the row exports)
        n1 = ctx.launch_count()
        ctx.slam_run_dev(d_frames[1].data_ptr(), k, deltas, z, pp, pe, ps)
        ctx.synchronize()
        assert ctx.launch_count() == n1 + k + 1
        assert (out.get()[2][:, 0, 0] >= 0).all()
        # the frames are the caller's: no resident frame is left for nav_slam_mapping(pos, NULL)
        with pytest.raises(pkg.NavError, match="no cloud is resident"):
            ctx.slam_mapping(z, None, want_global=False)
    finally:
        ctx.close()
