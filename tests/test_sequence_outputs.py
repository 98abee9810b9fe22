"""nav_frontend_sequence_out_dev: a device-resident sequence replay that keeps every frame's label masks, nn_idx,
nn_dist and fit totals instead of only the last frame's.

Every slot is held to the oracle driven along the same pose chain (labels, indices and distances bit for bit), the
fit totals to nav_slam_fit_stats of a second context stepped through the closed loop over the same frames (bit for
bit) and to exact sums of the oracle's correspondence list, and the context to the state nav_frontend_sequence_dev
leaves.  The cases cover the single-launch path (poses inline and through the device pose ring), the per-frame
path (several sequences, rows wider than 2048 columns, one frame, the profiler), ragged shapes, and motions whose
matches cross the tiles of a row."""
import ctypes as C
import importlib

import numpy as np
import pytest

from test_closed_loop_exact import check_stats, fit_py, tie_frames

gpu = pytest.mark.gpu
STEP = np.array([46.0, 2.0, -1.0, 0.0, 0.0, 0.0])
CANARY = 0xA5


# ------------------------------------------------------------------ helpers ----------------------------------
def seq_frames(synth, shape, n_seq, n, motion):
    """[n][n_seq][rows][cols][3]; 'scrambled' permutes every frame's columns, so a query's neighbour sits in an
    arbitrary tile of the row; 'empty_row' zeroes the middle row of every even frame, so the labelled queries of
    that row in the next frame search an empty map row (nn_idx -1, nn_dist +inf)."""
    r, c = shape
    fr = np.stack([np.stack([synth.room_frame(r, c, f, seq=s) for s in range(n_seq)]) for f in range(n)])
    if motion == "scrambled":
        rng = np.random.default_rng(r * 7919 + c)
        for f in range(n):
            for s in range(n_seq):
                fr[f, s] = fr[f, s][:, rng.permutation(c)]
    if motion == "empty_row":
        fr[::2, :, r // 2] = 0.0
    return np.ascontiguousarray(fr)


def pose_chain(k, n_seq, motion):
    """pred, last, final [k][n_seq][6] for frames 1..k; frame 0 is mapped at zero.  'large' turns 30 degrees of
    yaw per frame."""
    step = STEP + (np.array([0, 0, 0, 0, 0, 30.0]) if motion == "large" else 0.0)
    final = np.array([[(f + 1) * step + np.array([0.0, 0.5 * s, 0, 0, 0, 0]) for s in range(n_seq)] for f in range(k)])
    last = np.concatenate([np.zeros((1, n_seq, 6)), final[:-1]])
    pred = last + step + np.array([1.0, -0.5, 0.0, 0.0, 0.0, 0.1])
    return pred, last, final


def n_chunks(c):
    return -(-c // 16)


def unpack_mask(words, c):
    w = np.asarray(words).view(np.uint32)
    bits = (w[..., None] >> np.arange(16, dtype=np.uint32)) & 1
    return bits.reshape(w.shape[:-1] + (-1,))[..., :c].astype(np.int32)


_CUDART = None


def dev_to_numpy(p, dtype, count):
    """Copy `count` elements from a raw device pointer (buffers the context owns) to numpy."""
    global _CUDART
    if _CUDART is None:
        _CUDART = C.CDLL("libcudart.so")
    out = np.empty(count, dtype=dtype)
    rc = _CUDART.cudaMemcpy(C.c_void_p(out.ctypes.data), C.c_void_p(p), C.c_size_t(out.nbytes), C.c_int(2))
    assert rc == 0, rc
    return out


class Rings:
    """The four output buffers of k frames, each with guard bands filled with a canary on both sides."""
    GUARD = 4096   # bytes

    def __init__(self, torch, k, n_seq, r, c):
        self.torch = torch
        self.spec = {"label_mask": (np.uint32, (k, n_seq, r, n_chunks(c))), "nn_idx": (np.int32, (k, n_seq, r, c)),
                     "nn_dist": (np.float64, (k, n_seq, r, c)), "fit_stats": (np.float64, (k, n_seq, 5))}
        self.buf = {}
        for name, (dt, shp) in self.spec.items():
            nb = int(np.prod(shp)) * np.dtype(dt).itemsize
            self.buf[name] = torch.full((nb + 2 * self.GUARD,), CANARY, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()

    def ptr(self, name):
        return self.buf[name].data_ptr() + self.GUARD

    def ptrs(self, names):
        return {n: self.ptr(n) for n in names}

    def raw(self, name):
        return self.buf[name].cpu().numpy()

    def get(self, name):
        dt, shp = self.spec[name]
        return self.raw(name)[self.GUARD:-self.GUARD].view(dt).reshape(shp)

    def guards_intact(self, name):
        b = self.raw(name)
        return bool((b[:self.GUARD] == CANARY).all() and (b[-self.GUARD:] == CANARY).all())

    def untouched(self, name):
        return bool((self.raw(name) == CANARY).all())


def ctx_state(pkg, ctx, rows_to_export=(0,)):
    """Everything nav_frame_results_dev exposes plus a few rows of the map, copied to the host."""
    ctx.synchronize()
    res = ctx.frame_results_dev()
    n = ctx.n_seq * ctx.rows * ctx.cols
    st = {"labels": dev_to_numpy(res.labels, np.int32, n), "nn_idx": dev_to_numpy(res.nn_idx, np.int32, n),
          "nn_dist": dev_to_numpy(res.nn_dist, np.float64, n), "global": dev_to_numpy(res.global_, np.float64, 3 * n),
          "map_mask": dev_to_numpy(res.map_mask, np.uint32, ctx.n_seq * ctx.rows * n_chunks(ctx.cols))}
    for s in range(ctx.n_seq):
        for row in rows_to_export:
            st[f"row{s}.{row}"] = ctx.row_map_export(row, seq=s)
    return st


def assert_same_state(a, b):
    assert a.keys() == b.keys()
    for k in a:
        if isinstance(a[k], tuple):
            for x, y in zip(a[k], b[k]):
                assert x.tobytes() == y.tobytes(), k
        else:
            assert a[k].tobytes() == b[k].tobytes(), k


def replay(pkg, torch, shape, n_seq, d_frames, pred, last, final, rings=None, names=(), profile=False):
    """A fresh context mapped at frame 0, then the replay of frames 1..k with the named outputs."""
    r, c = shape
    k = pred.shape[0]
    ctx = pkg.Context(r, c, device=0, n_seq=n_seq)
    if profile:
        ctx.profile_enable(True)
    ctx.slam_init_dev(d_frames[0].data_ptr(), np.zeros((n_seq, 6)))
    ptrs = rings.ptrs(names) if rings is not None else {}
    n0 = ctx.launch_count()
    ctx.frontend_sequence_out_dev(d_frames[1].data_ptr(), k, pred.reshape(-1, 6), last.reshape(-1, 6),
                                  final.reshape(-1, 6), **ptrs)
    ctx.synchronize()
    return ctx, ctx.launch_count() - n0


# ------------------------------------------------------------------ 1 + 2: every frame, fit totals --------------
CASES = [((64, 2048), 1, 12), ((64, 2048), 1, 70), ((16, 1800), 1, 9), ((5, 33), 1, 6), ((3, 257), 1, 5),
         ((16, 1800), 3, 5), ((2, 4100), 1, 6), ((5, 33), 1, 1)]


@gpu
@pytest.mark.parametrize("shape,n_seq,k", CASES)
@pytest.mark.parametrize("motion", ["small", "large", "scrambled", "empty_row"])
def test_every_frame_matches_oracle_and_closed_loop(pkg, oracle, synth, shape, n_seq, k, motion):
    """Slot f against the oracle's frontend_frame of frame f (labels from the mask, nn_idx / nn_dist bit for bit
    on labelled pixels, -1 / -1.0 elsewhere); fit totals against a second single-sequence context stepped with
    nav_slam_localization_fast + nav_slam_mapping(final[f]) (bit for bit) and against exact sums of the oracle's
    correspondences; the host fit of the totals against fit_py and the pose that closed-loop call returned."""
    torch = pytest.importorskip("torch")
    r, c = shape
    frames = seq_frames(synth, shape, n_seq, k + 1, motion)
    pred, last, final = pose_chain(k, n_seq, motion)
    d_frames = torch.from_numpy(frames).cuda()
    rings = Rings(torch, k, n_seq, r, c)
    ctx, _ = replay(pkg, torch, shape, n_seq, d_frames, pred, last, final, rings, rings.spec.keys())
    ctx.close()
    mask, idx, dist, stats = (rings.get(n) for n in ("label_mask", "nn_idx", "nn_dist", "fit_stats"))
    for name in rings.spec:
        assert rings.guards_intact(name), name
    z = np.zeros(6)
    for s in range(n_seq):
        slam = oracle.slam(r, c, 1)
        loop = pkg.Context(r, c, device=0)
        try:
            slam.init(z, frames[0, s])
            loop.slam_init(z, frames[0, s], want_global=False)
            for f in range(k):
                cloud = frames[f + 1, s]
                _, corr, _, _ = slam.localize(cloud, pred[f, s], last[f, s])
                ofeat, oidx, odist, _ = slam.frontend_frame(cloud, pred[f, s], last[f, s], final[f, s])
                lab = ofeat == 1
                assert np.array_equal(unpack_mask(mask[f, s], c), ofeat), (f, s)
                assert np.array_equal(idx[f, s][lab], oidx[lab]), (f, s)
                assert dist[f, s][lab].tobytes() == odist[lab].tobytes(), (f, s)
                assert (idx[f, s][~lab] == -1).all() and (dist[f, s][~lab] == -1.0).all(), (f, s)
                if motion == "empty_row" and f % 2 == 0:  # frame f + 1 searched the empty row of frame f's map
                    q = lab[r // 2]
                    assert q.any() and (idx[f, s][r // 2][q] == -1).all(), (f, s)
                    assert (dist[f, s][r // 2][q] == np.inf).all(), (f, s)
                # the closed loop on the same map: localization_fast, then the map of the frame at final[f]
                p, err, nc = loop.slam_localization_fast(cloud, pred[f, s], last[f, s])
                st = stats[f, s]
                assert st.tobytes() == loop.slam_fit_stats().tobytes(), (f, s, st, loop.slam_fit_stats())
                loop.slam_mapping(final[f, s], None, want_global=False)
                check_stats(st, corr, shape)
                want, want_err, want_n = fit_py(st, pred[f, s], last[f, s])
                assert np.array_equal(p, want) and err == want_err and nc == want_n
                got, got_err = pkg.fit_from_stats(st, pred[f, s], last[f, s])
                assert np.array_equal(got, p) and got_err == err
        finally:
            loop.close()
            slam.close()


@gpu
@pytest.mark.parametrize("shape", [(3, 256), (3, 2048), (3, 4100)])
def test_fit_totals_exact_on_ties(pkg, oracle, synth, shape):
    """tie_frames: every residual an integer, so N, sum r and sum |r|^2 are exact -- a different dedupe winner of
    any tie would change them.  Both paths (one launch; rows wider than 2048 columns frame by frame)."""
    torch = pytest.importorskip("torch")
    r, c = shape
    A, B = tie_frames(synth, shape)
    frames = np.stack([A, B, A])[:, None]
    z = np.zeros((1, 6))
    pred = np.array([[[46.0, 2.0, -1.0, 0.0, 0.0, 0.0]]] * 2)
    last = np.zeros((2, 1, 6))
    final = np.zeros((2, 1, 6))
    d_frames = torch.from_numpy(np.ascontiguousarray(frames)).cuda()
    rings = Rings(torch, 2, 1, r, c)
    ctx, _ = replay(pkg, torch, shape, 1, d_frames, pred, last, final, rings, ["fit_stats"])
    ctx.close()
    stats = rings.get("fit_stats")
    slam = oracle.slam(r, c, 1)
    try:
        slam.init(z[0], A)
        for f in range(2):
            _, corr, _, _ = slam.localize(frames[f + 1, 0], pred[f, 0], last[f, 0])
            assert corr.shape[0] > 0
            check_stats(stats[f, 0], corr, shape, exact=True)
            slam.map(final[f, 0], frames[f + 1, 0])
    finally:
        slam.close()


# ------------------------------------------------------------------ 3: context state --------------------------
@gpu
@pytest.mark.parametrize("shape,n_seq,k", [((64, 2048), 1, 12), ((64, 2048), 1, 67), ((3, 257), 1, 5),
                                           ((16, 1800), 3, 4), ((2, 4100), 1, 5)])
def test_context_state_as_after_sequence_dev(pkg, synth, shape, n_seq, k):
    """After the call the context is byte for byte what nav_frontend_sequence_dev leaves (results, map, row
    exports), the next replay and a closed-loop step give the same results, and the last slot equals the
    context's buffers."""
    torch = pytest.importorskip("torch")
    r, c = shape
    frames = seq_frames(synth, shape, n_seq, k + 3, "large")
    pred, last, final = pose_chain(k + 2, n_seq, "large")
    d_frames = torch.from_numpy(frames).cuda()
    rings = Rings(torch, k, n_seq, r, c)
    rows = sorted({0, r // 2, r - 1})
    a, _ = replay(pkg, torch, shape, n_seq, d_frames, pred[:k], last[:k], final[:k], rings, rings.spec.keys())
    b, _ = replay(pkg, torch, shape, n_seq, d_frames, pred[:k], last[:k], final[:k])
    try:
        sa, sb = ctx_state(pkg, a, rows), ctx_state(pkg, b, rows)
        assert_same_state(sa, sb)
        assert rings.get("nn_idx")[-1].tobytes() == sa["nn_idx"].tobytes()
        assert rings.get("nn_dist")[-1].tobytes() == sa["nn_dist"].tobytes()
        assert rings.get("label_mask")[-1].tobytes() == sa["map_mask"].tobytes()
        assert np.array_equal(unpack_mask(rings.get("label_mask")[-1], c).reshape(-1), sa["labels"])
        # the next replay (one frame) continues from the same state
        for ctx in (a, b):
            ctx.frontend_sequence_dev(d_frames[k + 1].data_ptr(), 1, pred[k], last[k], final[k])
        assert_same_state(ctx_state(pkg, a, rows), ctx_state(pkg, b, rows))
        if n_seq == 1:   # and so does the closed loop
            ra = a.slam_localization_fast(frames[k + 2, 0], pred[k + 1, 0], last[k + 1, 0])
            rb = b.slam_localization_fast(frames[k + 2, 0], pred[k + 1, 0], last[k + 1, 0])
            assert np.array_equal(ra[0], rb[0]) and ra[1:] == rb[1:]
            assert a.slam_fit_stats().tobytes() == b.slam_fit_stats().tobytes()
    finally:
        a.close()
        b.close()


# ------------------------------------------------------------------ 4: null and partial outputs ---------------
@gpu
@pytest.mark.parametrize("shape,k", [((64, 2048), 12), ((2, 4100), 4)])
def test_null_outputs_are_sequence_dev(pkg, synth, shape, k):
    """out == NULL and a nav_sequence_out with every field NULL: the results and the launch count of
    nav_frontend_sequence_dev."""
    torch = pytest.importorskip("torch")
    r, c = shape
    frames = seq_frames(synth, shape, 1, k + 1, "small")
    pred, last, final = pose_chain(k, 1, "small")
    d_frames = torch.from_numpy(frames).cuda()
    L = pkg.load_library()
    binding = importlib.import_module("nav-slam_b200.binding")
    states, counts = [], []
    for how in ("sequence_dev", "out_null", "fields_null"):
        ctx = pkg.Context(r, c, device=0)
        try:
            ctx.slam_init_dev(d_frames[0].data_ptr(), np.zeros(6))
            n0 = ctx.launch_count()
            args = (d_frames[1].data_ptr(), k, binding._pos_array(pred.reshape(-1, 6), k),
                    binding._pos_array(last.reshape(-1, 6), k), binding._pos_array(final.reshape(-1, 6), k))
            if how == "sequence_dev":
                rc = L.nav_frontend_sequence_dev(ctx.h, *args)
            elif how == "out_null":
                rc = L.nav_frontend_sequence_out_dev(ctx.h, *args, None)
            else:
                rc = L.nav_frontend_sequence_out_dev(ctx.h, *args, C.byref(binding.NavSequenceOut()))
            assert rc == 0, L.nav_last_error()
            counts.append(ctx.launch_count() - n0)
            states.append(ctx_state(pkg, ctx, (0, r - 1)))
        finally:
            ctx.close()
    assert counts[0] == counts[1] == counts[2], counts
    assert_same_state(states[0], states[1])
    assert_same_state(states[0], states[2])


@gpu
@pytest.mark.parametrize("shape,k", [((1, 5), 4), ((3, 257), 5), ((2, 4100), 4)])
def test_each_field_alone_and_guard_bands(pkg, synth, shape, k):
    """Each field requested alone equals that field of the full call; nothing is written outside a requested
    slot range (canary guard bands), and buffers of fields that were not requested stay untouched."""
    torch = pytest.importorskip("torch")
    r, c = shape
    frames = seq_frames(synth, shape, 1, k + 1, "scrambled")
    pred, last, final = pose_chain(k, 1, "scrambled")
    d_frames = torch.from_numpy(frames).cuda()
    full = Rings(torch, k, 1, r, c)
    ctx, _ = replay(pkg, torch, shape, 1, d_frames, pred, last, final, full, full.spec.keys())
    ctx.close()
    for name in full.spec:
        assert full.guards_intact(name), name
        assert not full.untouched(name), name
    for name in full.spec:
        one = Rings(torch, k, 1, r, c)
        ctx, _ = replay(pkg, torch, shape, 1, d_frames, pred, last, final, one, [name])
        ctx.close()
        assert one.guards_intact(name), name
        assert one.get(name).tobytes() == full.get(name).tobytes(), name
        for other in full.spec:
            if other != name:
                assert one.untouched(other), (name, other)


# ------------------------------------------------------------------ 5 + 6: paths and launch counts ------------
@gpu
def test_fused_and_per_frame_paths_give_the_same_bytes(pkg, synth):
    """64x2048, 12 frames: the single launch and the per-frame path (forced by the profiler) fill every ring with
    the same bytes, and leave the same context state."""
    torch = pytest.importorskip("torch")
    shape, k = (64, 2048), 12
    r, c = shape
    frames = seq_frames(synth, shape, 1, k + 1, "scrambled")
    pred, last, final = pose_chain(k, 1, "scrambled")
    d_frames = torch.from_numpy(frames).cuda()
    got = []
    for profile in (False, True):
        rings = Rings(torch, k, 1, r, c)
        ctx, launches = replay(pkg, torch, shape, 1, d_frames, pred, last, final, rings, rings.spec.keys(),
                               profile=profile)
        got.append(({n: rings.get(n).tobytes() for n in rings.spec}, ctx_state(pkg, ctx, (0, 31, 63)), launches))
        ctx.close()
    assert got[0][2] == 2 and got[1][2] == 2 * k + 1, (got[0][2], got[1][2])
    for n in got[0][0]:
        assert got[0][0][n] == got[1][0][n], n
    assert_same_state(got[0][1], got[1][1])


@gpu
@pytest.mark.parametrize("k", [12, 40])
def test_launch_count_of_the_single_launch_path(pkg, synth, k):
    torch = pytest.importorskip("torch")
    shape = (64, 2048)
    r, c = shape
    frames = seq_frames(synth, shape, 1, k + 1, "small")
    pred, last, final = pose_chain(k, 1, "small")
    d_frames = torch.from_numpy(frames).cuda()
    rings = Rings(torch, k, 1, r, c)
    for names, want in (((), 1), (("label_mask", "nn_idx", "nn_dist"), 1), (("fit_stats",), 2),
                        (tuple(rings.spec), 2)):
        ctx, launches = replay(pkg, torch, shape, 1, d_frames, pred, last, final, rings, names)
        ctx.close()
        assert launches == want, (names, launches)


# ------------------------------------------------------------------ 7: the host fit ---------------------------
def test_fit_from_stats_matches_the_python_restatement(pkg):
    """CPU only: nav_slam_fit_from_stats against fit_py on hand-made totals, including N = 0 (the pose stays at
    the prediction as last + (pred - last), error 0)."""
    pred = np.array([51.25, -3.5, 0.75, 0.5, -0.25, 2.0])
    last = np.array([1.0, -0.5, 0.25, 0.0, 0.0, 1.5])
    cases = [np.zeros(5), np.array([1.0, 50.0, -3.0, 0.5, 2509.25]),
             np.array([4211.0, 2.1e5, -1.2e4, 2.2e3, 1.3e7]), np.array([17.0, -851.0, 35.5, -15.0, 4.4e4])]
    for st in cases:
        want, want_err, _ = fit_py(st, pred, last)
        got, err = pkg.fit_from_stats(st, pred, last)
        assert np.array_equal(got, want) and err == want_err, (st, got - want, err, want_err)
    got, err = pkg.fit_from_stats(np.zeros(5), pred, last)
    assert np.array_equal(got, last + (pred - last)) and err == 0.0
    L = pkg.load_library()   # the binding always passes every argument: the C guard directly
    assert L.nav_slam_fit_from_stats(None, None, None, None, None) != 0
    assert b"null argument" in L.nav_last_error()


# ------------------------------------------------------------------ 8: rejected input, default stream ---------
@gpu
@pytest.mark.parametrize("field", ["label_mask", "nn_idx", "nn_dist", "fit_stats"])
def test_host_pointer_is_rejected_by_name(pkg, synth, field):
    torch = pytest.importorskip("torch")
    shape, k = (3, 257), 3
    r, c = shape
    frames = seq_frames(synth, shape, 1, k + 1, "small")
    pred, last, final = pose_chain(k, 1, "small")
    d_frames = torch.from_numpy(frames).cuda()
    rings = Rings(torch, k, 1, r, c)
    host = np.zeros(k * r * c * 8 + 4096, dtype=np.uint8)
    L = pkg.load_library()
    pinned = L.nav_host_alloc(host.nbytes)
    ctx = pkg.Context(r, c, device=0)
    try:
        ctx.slam_init_dev(d_frames[0].data_ptr(), np.zeros(6))
        for bad in (host.ctypes.data, pinned):
            ptrs = rings.ptrs(rings.spec.keys())
            ptrs[field] = bad
            n0 = ctx.launch_count()
            with pytest.raises(pkg.NavError, match=field):
                ctx.frontend_sequence_out_dev(d_frames[1].data_ptr(), k, pred.reshape(-1, 6), last.reshape(-1, 6),
                                              final.reshape(-1, 6), **ptrs)
            assert ctx.launch_count() == n0
        ctx.synchronize()
        for name in rings.spec:
            assert rings.untouched(name), name
    finally:
        ctx.close()
        L.nav_host_free(pinned)


@gpu
def test_replay_on_the_legacy_default_stream(pkg, synth):
    """set_stream(0): the same outputs as on the context's own stream once the device is synchronised."""
    torch = pytest.importorskip("torch")
    shape, k = (16, 1800), 6
    r, c = shape
    frames = seq_frames(synth, shape, 1, k + 1, "large")
    pred, last, final = pose_chain(k, 1, "large")
    d_frames = torch.from_numpy(frames).cuda()
    ref = Rings(torch, k, 1, r, c)
    ctx, _ = replay(pkg, torch, shape, 1, d_frames, pred, last, final, ref, ref.spec.keys())
    ctx.close()
    rings = Rings(torch, k, 1, r, c)
    ctx = pkg.Context(r, c, device=0)
    try:
        ctx.set_stream(0)
        ctx.slam_init_dev(d_frames[0].data_ptr(), np.zeros(6))
        ctx.frontend_sequence_out_dev(d_frames[1].data_ptr(), k, pred.reshape(-1, 6), last.reshape(-1, 6),
                                      final.reshape(-1, 6), **rings.ptrs(rings.spec.keys()))
        torch.cuda.synchronize()
        for n in ref.spec:
            assert rings.get(n).tobytes() == ref.get(n).tobytes(), n
    finally:
        ctx.close()
