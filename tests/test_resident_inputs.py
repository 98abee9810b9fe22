"""Depth and integer-mm recordings in the device-resident calls: nav_slam_init_dev_ex, nav_frontend_sequence_dev_ex
and nav_slam_run_dev_ex take the frames as the sensors give them and convert them inside the kernels.

Each call is held bit for bit to its xyz form on the clouds the frames stand for -- every ring of the replay, the
poses, errors and fit totals of the closed loop, and the context afterwards -- on every staging path of the sequence
kernel (bulk copies, 4-byte cp.async, one launch per frame), and independently of the xyz path to the oracle.  The
frames carry dropouts (zero and negative depths, scattered and in whole tiles) and integer-mm extremes (+-(2^31-1),
zero, negative coordinates)."""
import importlib

import numpy as np
import pytest

from test_closed_loop_exact import check_stats, pinned, ptr
from test_seq_bulk_staging import sequence_path
from test_sequence_outputs import Rings, assert_same_state, ctx_state, pose_chain, unpack_mask
from test_slam_run_dev import DevOut, deltas_of, same_values

gpu = pytest.mark.gpu
DEPTH, MM = "depth", "mm"
I32_MAX = 2 ** 31 - 1


# ------------------------------------------------------------------ generators ------------------------------------
def room(synth, shape, n, n_seq, integer_mm=False):
    r, c = shape
    return np.stack([np.stack([synth.room_frame(r, c, f, seq=s, integer_mm=integer_mm) for s in range(n_seq)])
                     for f in range(n)])


def depth_frames(synth, shape, n, n_seq=1):
    """int32 [n][n_seq][rows][cols]: the room ranges as bench.py forms them, with dropouts -- zero and negative
    depths in scattered pixels, and whole 256-column tiles of zeros / negatives in some frames."""
    r, c = shape
    d = np.clip(np.linalg.norm(room(synth, shape, n, n_seq), axis=-1), 1, 60000).astype(np.int32)
    rng = np.random.default_rng(r * 31 + c)
    hole = rng.random(d.shape) < 0.01
    d[hole] = rng.choice(np.array([0, -1, -60000, np.iinfo(np.int32).min], dtype=np.int32), int(hole.sum()))
    for f in range(1, n, 3):
        d[f, :, (f * 7) % r, :min(c, 256)] = 0
        d[f, :, (f * 5 + 1) % r, max(0, c - 300):] = -3
    return np.ascontiguousarray(d)


def mm_frames(synth, pkg, shape, n, n_seq=1):
    """int32 [n][n_seq][rows][cols][3]: binding.to_mm of the integer-mm room, with coordinates of +-(2^31-1), zero and
    negative values in scattered pixels."""
    m = pkg.to_mm(room(synth, shape, n, n_seq, integer_mm=True) + 0.0)   # + 0.0: no -0.0, which to_mm refuses
    rng = np.random.default_rng(shape[0] * 17 + shape[1])
    flat = m.reshape(-1, 3)
    idx = rng.choice(flat.shape[0], max(4, flat.shape[0] // 500), replace=False)
    vals = np.array([I32_MAX, -I32_MAX, 0, -1, -123456], dtype=np.int32)
    flat[idx] = rng.choice(vals, (idx.size, 3))
    return np.ascontiguousarray(m)


def to_xyz(pkg, kind, raw):
    """The clouds the frames stand for: nav_convert_to_pointcloud of every depth image, float64 of the mm values."""
    if kind == MM:
        return raw.astype(np.float64)
    r, c = raw.shape[-2:]
    conv = pkg.Context(r, c, device=0)
    try:
        out = np.stack([conv.convert_to_pointcloud(img) for img in raw.reshape(-1, r, c)])
    finally:
        conv.close()
    return np.ascontiguousarray(out.reshape(raw.shape + (3,)))


def frames_of(synth, pkg, kind, shape, n, n_seq=1):
    raw = depth_frames(synth, shape, n, n_seq) if kind == DEPTH else mm_frames(synth, pkg, shape, n, n_seq)
    return raw, to_xyz(pkg, kind, raw)


def kw(kind):
    return {"depth_input": kind == DEPTH, "mm_input": kind == MM}


def sequence(pkg, shape, n_seq, d0, d1, pred, last, final, rings, kind=None, ptr1=None):
    """A fresh context mapped at zero with frame d0, then the replay of d1 with every ring."""
    r, c = shape
    ctx = pkg.Context(r, c, device=0, n_seq=n_seq)
    args = kw(kind) if kind else {}
    ctx.slam_init_dev(d0.data_ptr(), np.zeros((n_seq, 6)), **args)
    n0 = ctx.launch_count()
    ctx.frontend_sequence_out_dev(ptr1 if ptr1 is not None else d1.data_ptr(), pred.shape[0], pred.reshape(-1, 6),
                                  last.reshape(-1, 6), final.reshape(-1, 6), **rings.ptrs(rings.spec.keys()), **args)
    ctx.synchronize()
    return ctx, ctx.launch_count() - n0


# ------------------------------------------------------------------ 1. replay parity --------------------------
# (shape, n_seq, frames, staging path of the narrow kinds: 2 bulk, 1 cp.async, 0 one launch per frame, offset bytes)
REPLAY = [((64, 2048), 1, 20, 2, 0), ((64, 2048), 1, 65, 2, 0), ((4, 192), 1, 6, 2, 0), ((4, 768), 1, 6, 2, 0),
          ((16, 1800), 1, 8, 1, 0), ((5, 258), 1, 6, 1, 0), ((64, 2048), 1, 6, 1, 4), ((16, 1800), 3, 5, 0, 0),
          ((2, 4100), 1, 5, 0, 0)]


@gpu
@pytest.mark.parametrize("kind", [DEPTH, MM])
@pytest.mark.parametrize("shape,n_seq,k,path,offset", REPLAY)
def test_replay_equals_the_xyz_replay(pkg, synth, kind, shape, n_seq, k, path, offset):
    """nav_frontend_sequence_dev_ex with all four rings against nav_frontend_sequence_out_dev on the converted frames:
    every slot, then nav_frame_results_dev and several exported map rows, bit for bit; the staging path taken."""
    torch = pytest.importorskip("torch")
    r, c = shape
    raw, xyz = frames_of(synth, pkg, kind, shape, k + 1, n_seq)
    pred, last, final = pose_chain(k, n_seq, "small")
    d_raw, d_xyz = torch.from_numpy(raw).cuda(), torch.from_numpy(xyz).cuda()
    ptr1 = None
    if offset:  # the frames 4 bytes past a 16-byte boundary
        flat = torch.zeros(raw[1:].size + 4, dtype=torch.int32, device="cuda")
        flat[1:1 + raw[1:].size] = d_raw[1:].reshape(-1)
        ptr1 = flat.data_ptr() + offset
        assert ptr1 % 16 == offset
    ring_a, ring_b = Rings(torch, k, n_seq, r, c), Rings(torch, k, n_seq, r, c)
    a, na = sequence(pkg, shape, n_seq, d_raw[0], d_raw[1], pred, last, final, ring_a, kind, ptr1)
    b, nb = sequence(pkg, shape, n_seq, d_xyz[0], d_xyz[1], pred, last, final, ring_b)
    try:
        assert sequence_path(pkg, a) == path
        # the per-frame path converts each frame first: one more launch per frame
        assert na == nb + (k if path == 0 else 0), (na, nb)
        for name in ring_a.spec:
            assert ring_a.guards_intact(name), name
            assert ring_a.get(name).tobytes() == ring_b.get(name).tobytes(), name
        rows = sorted({0, 1 % r, r // 2, r - 1})
        assert_same_state(ctx_state(pkg, a, rows), ctx_state(pkg, b, rows))
    finally:
        a.close()
        b.close()


# ------------------------------------------------------------------ 2. against the oracle ---------------------
@gpu
def test_depth_replay_against_the_oracle(pkg, oracle, synth):
    """A 64x2048 depth replay of 12 frames walked with oracle.convert and the oracle's frame step: labels, nn_idx and
    nn_dist bit for bit, fit totals against exact sums of the oracle's correspondences."""
    torch = pytest.importorskip("torch")
    shape, k = (64, 2048), 12
    r, c = shape
    raw = depth_frames(synth, shape, k + 1)
    pred, last, final = pose_chain(k, 1, "small")
    d_raw = torch.from_numpy(raw).cuda()
    rings = Rings(torch, k, 1, r, c)
    ctx, _ = sequence(pkg, shape, 1, d_raw[0], d_raw[1], pred, last, final, rings, DEPTH)
    try:
        assert sequence_path(pkg, ctx) == 2
    finally:
        ctx.close()
    mask, idx, dist, stats = (rings.get(n)[:, 0] for n in ("label_mask", "nn_idx", "nn_dist", "fit_stats"))
    slam = oracle.slam(r, c, 1)
    try:
        slam.init(np.zeros(6), oracle.convert(raw[0, 0]))
        for f in range(k):
            cloud = oracle.convert(raw[f + 1, 0])
            _, corr, _, _ = slam.localize(cloud, pred[f, 0], last[f, 0])
            ofeat, oidx, odist, _ = slam.frontend_frame(cloud, pred[f, 0], last[f, 0], final[f, 0])
            lab = ofeat == 1
            assert np.array_equal(unpack_mask(mask[f], c), ofeat), f
            assert np.array_equal(idx[f][lab], oidx[lab]), f
            assert dist[f][lab].tobytes() == odist[lab].tobytes(), f
            assert (idx[f][~lab] == -1).all() and (dist[f][~lab] == -1.0).all(), f
            check_stats(stats[f], corr, shape)
    finally:
        slam.close()


# ------------------------------------------------------------------ 3. closed loop -----------------------------
def dev_run(pkg, torch, shape, raw, deltas, start, kind):
    """nav_slam_run_dev[_ex] on a fresh context mapped at start with frame 0 (kind None: xyz frames)."""
    r, c = shape
    k, n_seq = raw.shape[0] - 1, raw.shape[1]
    ctx = pkg.Context(r, c, device=0, n_seq=n_seq)
    d = torch.from_numpy(raw).cuda()
    args = kw(kind) if kind else {}
    ctx.slam_init_dev(d[0].data_ptr(), start.reshape(n_seq, 6), **args)
    out = DevOut(torch, k, n_seq)
    n0 = ctx.launch_count()
    ctx.slam_run_dev(d[1].data_ptr(), k, deltas.reshape(-1, 6), start.reshape(n_seq, 6), *out.ptrs(), **args)
    ctx.synchronize()
    assert ctx.launch_count() - n0 == k + 1
    return ctx, out.get()


@gpu
@pytest.mark.parametrize("kind", [DEPTH, MM])
def test_closed_loop_equals_host_loop_and_xyz(pkg, synth, kind):
    """n_seq = 1: nav_slam_run_dev_ex equals nav_slam_run on the host frames of the same kind (poses, errors,
    correspondence counts) and nav_slam_run_dev on the converted frames (fit totals too), bit for bit."""
    torch = pytest.importorskip("torch")
    shape, k = (64, 2048), 10
    r, c = shape
    raw, xyz = frames_of(synth, pkg, kind, shape, k + 1)
    deltas = deltas_of(k, 1, seed=5)
    start = np.zeros((1, 6))
    a, (pa, ea, sa) = dev_run(pkg, torch, shape, raw, deltas, start, kind)
    b, (pb, eb, sb) = dev_run(pkg, torch, shape, xyz, deltas, start, None)
    host = pkg.Context(r, c, device=0)
    try:
        assert same_values(pa, pb) and same_values(ea, eb) and same_values(sa, sb)
        assert_same_state(ctx_state(pkg, a, (0, r - 1)), ctx_state(pkg, b, (0, r - 1)))
        host.slam_init(start[0], xyz[0, 0], want_global=False)
        frames = np.ascontiguousarray(raw[1:, 0])
        with pinned(pkg, frames):
            poses, errs, ncs = host.slam_run([ptr(frames[f]) for f in range(k)], deltas[:, 0], start[0], **kw(kind))
        assert same_values(pa[:, 0], poses) and same_values(ea[:, 0], errs)
        assert np.array_equal(sa[:, 0, 0].astype(np.int64), ncs)
    finally:
        for x in (a, b, host):
            x.close()


@gpu
@pytest.mark.parametrize("kind", [DEPTH, MM])
@pytest.mark.parametrize("shape,n_seq", [((16, 1800), 3), ((8, 600), 16)])
def test_closed_loop_sequences_side_by_side(pkg, synth, kind, shape, n_seq):
    """Several sequences in the same launches: each equals a single-sequence run of itself."""
    torch = pytest.importorskip("torch")
    k = 5
    raw, _ = frames_of(synth, pkg, kind, shape, k + 1, n_seq)
    deltas = deltas_of(k, n_seq, seed=n_seq)
    start = np.array([[0.0, 300.0 * s, 0.0, 0.0, 0.0, 0.0] for s in range(n_seq)])
    ctx, (p, e, st) = dev_run(pkg, torch, shape, raw, deltas, start, kind)
    ctx.close()
    for s in range(n_seq):
        one, (p1, e1, st1) = dev_run(pkg, torch, shape, np.ascontiguousarray(raw[:, s:s + 1]), deltas[:, s:s + 1],
                                     start[s:s + 1], kind)
        one.close()
        assert same_values(p[:, s], p1[:, 0]) and same_values(e[:, s], e1[:, 0]) and same_values(st[:, s], st1[:, 0]), s


# ------------------------------------------------------------------ 4. init -----------------------------------
@gpu
@pytest.mark.parametrize("kind", [DEPTH, MM])
@pytest.mark.parametrize("shape,n_seq", [((64, 2048), 1), ((16, 1800), 3)])
def test_init_gives_the_map_of_the_converted_cloud(pkg, synth, kind, shape, n_seq):
    torch = pytest.importorskip("torch")
    r, c = shape
    raw, xyz = frames_of(synth, pkg, kind, shape, 1, n_seq)
    pos = np.array([[10.0 * s, -5.0, 2.0, 0.0, 0.0, 3.0 * s] for s in range(n_seq)])
    a = pkg.Context(r, c, device=0, n_seq=n_seq)
    b = pkg.Context(r, c, device=0, n_seq=n_seq)
    try:
        a.slam_init_dev(torch.from_numpy(raw[0]).cuda().data_ptr(), pos, **kw(kind))
        b.slam_init(pos if n_seq > 1 else pos[0], xyz[0] if n_seq > 1 else xyz[0, 0], want_global=False)
        sa, sb = ctx_state(pkg, a, (0, r // 2, r - 1)), ctx_state(pkg, b, (0, r // 2, r - 1))
        for name in ("nn_idx", "nn_dist"):   # what the init leaves there is not part of the map
            del sa[name], sb[name]
        assert_same_state(sa, sb)
    finally:
        a.close()
        b.close()


# ------------------------------------------------------------------ 5. mixed use ------------------------------
@gpu
def test_mixed_use_on_one_context(pkg, synth):
    """xyz replay, depth replay, integer-mm closed loop, then a host nav_slam_localization_fast, against the same
    calls on converted frames."""
    torch = pytest.importorskip("torch")
    shape, k = (64, 2048), 4
    r, c = shape
    xyz0 = room(synth, shape, k + 1, 1)
    draw, dxyz = frames_of(synth, pkg, DEPTH, shape, k + 1)
    mraw, mxyz = frames_of(synth, pkg, MM, shape, k + 1)
    pred, last, final = pose_chain(k, 1, "small")
    deltas = deltas_of(k, 1, seed=9)
    host = room(synth, shape, 1, 1)[0, 0]

    def run(depth, mm, depth_kw, mm_kw):
        ctx = pkg.Context(r, c, device=0)
        d0, dd, dm = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (xyz0, depth, mm))
        ctx.slam_init_dev(d0[0].data_ptr(), np.zeros(6))
        ctx.frontend_sequence_dev(d0[1].data_ptr(), k, pred.reshape(-1, 6), last.reshape(-1, 6), final.reshape(-1, 6))
        ctx.frontend_sequence_dev(dd[1].data_ptr(), k, pred.reshape(-1, 6), last.reshape(-1, 6), final.reshape(-1, 6),
                                  **depth_kw)
        out = DevOut(torch, k, 1)
        ctx.slam_run_dev(dm[1].data_ptr(), k, deltas.reshape(-1, 6), final[-1], *out.ptrs(), **mm_kw)
        ctx.synchronize()
        got = out.get()
        p, err, nc = ctx.slam_localization_fast(host, got[0][-1, 0] + np.array([40.0, 1.0, 0, 0, 0, 0]), got[0][-1, 0])
        state = ctx_state(pkg, ctx, (0, r - 1))
        ctx.close()
        return got, (p, err, nc), state

    ga, la, sa = run(draw, mraw, kw(DEPTH), kw(MM))
    gb, lb, sb = run(dxyz, mxyz, {}, {})
    for x, y in zip(ga, gb):
        assert same_values(x, y)
    assert same_values(la[0], lb[0]) and la[1:] == lb[1:]
    assert_same_state(sa, sb)


# ------------------------------------------------------------------ 6. refusals -------------------------------
@gpu
def test_refusals_name_their_cause_and_queue_nothing(pkg, synth):
    torch = pytest.importorskip("torch")
    import ctypes as C
    shape, k = (16, 256), 2
    r, c = shape
    raw, _ = frames_of(synth, pkg, DEPTH, shape, k + 1)
    d = torch.from_numpy(raw).cuda()
    ctx = pkg.Context(r, c, device=0)
    L = ctx.L
    NavPos = importlib.import_module("nav-slam_b200.binding").NavPos
    NavRunDevOut = importlib.import_module("nav-slam_b200.binding").NavRunDevOut
    try:
        ctx.slam_init_dev(d[0].data_ptr(), np.zeros(6), depth_input=True)
        ctx.synchronize()
        before_state = ctx_state(pkg, ctx, (0,))
        pos = (NavPos * k)()
        one = (NavPos * 1)()
        out = DevOut(torch, k, 1)
        dev_out = NavRunDevOut(*out.ptrs())
        host_out = np.zeros((k, 6))
        host_frames = np.ascontiguousarray(raw[1:])
        p1 = d[1].data_ptr()

        def seq(p, kind):
            return L.nav_frontend_sequence_dev_ex(ctx.h, p, kind, k, pos, pos, pos, None)

        def run(p, kind, o=dev_out):
            return L.nav_slam_run_dev_ex(ctx.h, p, kind, k, pos, one, C.byref(o))

        def init(p, kind):
            return L.nav_slam_init_dev_ex(ctx.h, p, kind, one)

        cases = [("input_kind 3", lambda: seq(p1, 3), "input_kind 3"),
                 ("input_kind -1", lambda: run(p1, -1), "input_kind -1"),
                 ("input_kind 7 init", lambda: init(p1, 7), "input_kind 7"),
                 ("2-byte offset seq", lambda: seq(p1 + 2, 1), "aligned"),
                 ("2-byte offset run", lambda: run(p1 + 2, 2), "aligned"),
                 ("2-byte offset init", lambda: init(p1 + 2, 1), "aligned"),
                 ("null frames", lambda: seq(None, 1), "null"),
                 ("null init", lambda: init(None, 2), "null"),
                 ("host frames", lambda: run(host_frames.ctypes.data, 1), "dev_frames"),
                 ("host output", lambda: run(p1, 1, NavRunDevOut(host_out.ctypes.data, None, None)), "out->poses")]
        for name, call, cause in cases:
            n0 = ctx.launch_count()
            assert call() != 0, name
            msg = L.nav_last_error().decode()
            assert cause in msg, (name, msg)
            assert ctx.launch_count() == n0, name
        ctx.set_tie_rule("reference")
        for name, call in [("seq", lambda: seq(p1, 1)), ("run", lambda: run(p1, 2))]:
            n0 = ctx.launch_count()
            assert call() != 0, name
            assert "tie rule" in L.nav_last_error().decode(), name
            assert ctx.launch_count() == n0, name
        ctx.set_tie_rule("lowest_index")
        assert_same_state(ctx_state(pkg, ctx, (0,)), before_state)
        with pytest.raises(ValueError):
            ctx.slam_run_dev(p1, k, np.zeros((k, 6)), np.zeros(6), *out.ptrs(), depth_input=True, mm_input=True)
    finally:
        ctx.close()
