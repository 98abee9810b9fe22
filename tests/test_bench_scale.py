"""Every workload bench.py times, run at the size it times it and held bit for bit to the reference.

The rest of the suite is thorough on shape edges but runs small inputs.  At the benchmark's sizes the kernels enter
regimes those never reach: the TMA ring of a persistent CTA wraps hundreds of times, grids span several resident
waves while programmatic dependent launch overlaps consecutive launches, per-sequence tickets and the "last CTA of
the sequence runs the fit" rule play out across many waves of clusters, and kd searches answer full query sets on
the maps a SLAM run produces.  Each test runs one bench leg at the bench's size (DESIGN.md section 7 names the row
that reports it):

* test_batch_labels_at_bench_size[512], [1000]: kernels.labels_batch, k_labels_tma on 512 images of 64x2048 (the
  default) and 1000 (config 3, 3.1 GB of input); row "curvature stencil, 512- / 1000-image batch".  Every CTA
  handles >= 100 tiles, so its 4-stage ring wraps >= 25 times.  [odd]: an odd point count at the same depth of
  wraps, so the hand-stored trailing double of the last tile comes after ~100 rounds.
* test_eight_sequences_replay: batched_sequences, config 5a on one GPU (8 sequences of 64x2048 side by side
  through nav_frontend_sequence_dev, 32 frames); row "8 sequences per launch".  4096 CTAs per k_frame_match
  launch, several resident waves, consecutive launches overlapped by programmatic dependent launch.
* test_eight_sequences_every_frame: nav_frontend_sequence_out_dev with 8 sequences (the per-frame path, rings and
  fit totals, profiles/prof_seq_outputs.py); row "replay keeping every frame's results", eight sequences.  The same
  grids plus k_dedupe_stats and the fit totals over 8 x 64 x 8 partials per frame.
* test_slam_run_dev_many_sequences[8], [16]: nav_slam_run_dev at 64x2048 (profiles/prof_slam_run_dev.py, 2 / 4 /
  8 sequences in README.md); row "closed loop on resident frames".  4096 / 8192 clustered k_loop_step<true> CTAs,
  per-sequence tickets across many waves of 8-CTA clusters.
* test_kd_tree_every_query[uniform_1m], [accumulated]: nn, config 4 (1 M uniform map with jittered and uniform
  queries, the accumulated room map of synth.accumulated_map(8) with the next frame's 131 072 points); rows
  "kd-tree queries, 131 072 vs ...".  [uniform_10m]: config 5b's 10 M-point map queried on one GPU (bench.py
  --big-map), a 24-level tree; row "10 M-point map".  Both split rules, every query.
* test_stackless_kd_kernels_every_query[plain], [conv]: the same maps through NAV_KD_KERNEL=plain|conv.
* test_tensor_cores_every_query[accumulated], [uniform_1m]: nn.tensor_core_bruteforce, config 4; row "config 4,
  same map and queries through the tensor-core tiles".  3907 / 4096 point tiles per CTA through the operand ring
  and a flag mask of up to 512 MB; the bench's same_answers_as_kdtree becomes an assertion.

The references: oracle.extract_feature for labels; the oracle's frontend_frame walked frame by frame (and localize
with check_stats for fit totals) for the sequence replays, together with single-sequence replays of each sequence
(a different kernel: k_frame_seq); nav_slam_run and single-sequence nav_slam_run_dev for the closed loop; the fp64
brute force k_bf_nn for every query of the map searches, itself held to oracle.nn_brute on 512 random queries of
every query set.  The launch arithmetic in each test shows that the bench's regime is reached: one 256-thread CTA
per tile, and at most max_threads_per_multi_processor / 256 of them resident on an SM.

The CPU side dominates the run time (the oracle's frontend_frame takes about 0.3 s per 64x2048 frame on one core);
it runs on a thread pool, one sequence or one block of images or queries per thread, since ctypes releases the
GIL.
"""
import concurrent.futures
import gc
import os
import subprocess
import sys
import tempfile
from types import SimpleNamespace

import numpy as np
import pytest

from test_closed_loop_exact import check_stats, pinned
from test_label_threshold import POISON, Guarded, bounds_of, counted, dev_to_numpy, near_threshold_images, ran
from test_sequence_outputs import Rings, pose_chain, replay, seq_frames, unpack_mask
from test_slam_run_dev import deltas_of, dev_loop, frames_of, host_loop, same_bits

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKERS = min(32, os.cpu_count() or 1)
CTA_THREADS = 256   # every kernel below: k_labels_tma, k_frame_match, k_loop_step (kTile)


# ------------------------------------------------------------------ helpers ----------------------------------
def pool_map(fn, items):
    with concurrent.futures.ThreadPoolExecutor(max_workers=WORKERS) as ex:
        return list(ex.map(fn, items))


def resident_wave(torch):
    """The most 256-thread CTAs the device holds at once (the thread limit of an SM times the SMs): no occupancy
    a kernel reaches can exceed it."""
    p = torch.cuda.get_device_properties(0)
    return p.multi_processor_count * (p.max_threads_per_multi_processor // CTA_THREADS)


def need_device(torch, nbytes, what):
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip(f"{what} needs {nbytes / 1e9:.1f} GB of device memory, {free / 1e9:.1f} GB free")


@pytest.fixture(autouse=True)
def _release_device_memory():
    """Each case frees its buffers before the next: the library allocates outside torch's cache."""
    yield
    gc.collect()
    torch = sys.modules.get("torch")
    if torch is not None and torch.cuda.is_initialized():
        torch.cuda.empty_cache()


def assert_nn(idx, dist, want_idx, want_dist, msg):
    assert np.array_equal(idx, want_idx), (msg, np.count_nonzero(idx != want_idx), np.nonzero(idx != want_idx)[0][:8])
    assert dist.tobytes() == want_dist.tobytes(), (msg, np.nonzero(dist != want_dist)[0][:8])


# ------------------------------------------------------------------ 1. batch labels --------------------------
K_TILE_OUT = 240   # output points per 1-D tile of k_labels_tma (stencil.cu: 8 warps x 30)
N_NEAR = 6         # near-threshold images mixed into every batch
CHUNK = 64         # images generated and uploaded at a time

# The kernel launch_labels picks for a batch depends only on the point count, the row width and the alignment of
# the cloud, so a process of its own makes the same call on zeros under torch's profiler (kernels_run) and prints
# the kernel names.  In the pytest process, a profiler session this early followed by the rest of the suite left
# later sessions (test_label_threshold.py) without kernel records.
KERNEL_PROBE = """
import importlib, sys
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import torch
from test_label_threshold import kernels_run
rows, cols, n, first = map(int, sys.argv[2:])
pkg = importlib.import_module("nav-slam_b200")
buf = torch.zeros(first + n * rows * cols * 3, dtype=torch.float64, device="cuda")
labels = torch.empty(n * rows * cols, dtype=torch.int32, device="cuda")
ctx = pkg.Context(rows, cols, device=0)
ctx.set_stream(torch.cuda.current_stream().cuda_stream)
_, names = kernels_run(torch, lambda: ctx.extract_feature_batch_dev(buf.data_ptr() + first * 8, n, labels.data_ptr()))
ctx.close()
print(names)
"""


def batch_kernels(rows, cols, n, first):
    """names of the kernels nav_extract_feature_batch_dev runs on n images of rows x cols at double offset first"""
    res = subprocess.run([sys.executable, "-c", KERNEL_PROBE, ROOT, str(rows), str(cols), str(n), str(first)],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    return res.stdout


def batch_images(synth, shape, n):
    """image(i) of a batch of n distinct images: room frames of different frames and sequences (every one with its
    own noise), with N_NEAR near-threshold images at the first, the last and evenly spaced positions.  A tile fed
    from a stale or wrong ring slot then changes labels."""
    at = np.linspace(0, n - 1, N_NEAR).round().astype(int)
    near = dict(zip(at.tolist(), near_threshold_images(shape, N_NEAR, 900 + n)))

    def image(i):
        return near[i] if i in near else synth.room_frame(*shape, i % 100, seq=i // 100)
    return image, list(near.values())


@gpu
@pytest.mark.parametrize("shape,n", [((64, 2048), 512), ((64, 2048), 1000), ((33, 1001), 861)],
                         ids=["512", "1000", "odd"])
def test_batch_labels_at_bench_size(pkg, oracle, synth, shape, n):
    """nav_extract_feature_batch_dev on the bench's batches (512 and 1000 images of 64x2048) and on an odd point
    count at the same depth of ring wraps (861 images of 33x1001: the last bulk copy ends on a hand-stored double).
    The batch sits between NaN points and the labels between canary guard bands, as in test_batch_labels; every
    label is held to oracle.extract_feature, and the exact re-evaluations to at least those the near-threshold
    images force.  The same call in a process of its own (batch_kernels) runs k_labels_tma."""
    torch = pytest.importorskip("torch")
    rows, cols = shape
    npx = rows * cols
    n_pts = n * npx
    # launch arithmetic of launch_labels: k_labels_tma for >= 4 tiles per SM, one resident wave of CTAs, each
    # taking every grid-th tile -- so every CTA handles at least n_tiles_1d // (one resident wave) tiles
    n_tiles_1d = -(-n_pts // K_TILE_OUT)
    wave = resident_wave(torch)
    assert n_tiles_1d >= 4 * torch.cuda.get_device_properties(0).multi_processor_count and n_pts < 2 ** 31
    assert n_tiles_1d // wave >= 100, (n_tiles_1d, wave)
    if shape == (33, 1001):
        assert n_pts % 2 == 1   # the last tile holds an odd number of points: 8 bytes past the bulk copy
    need_device(torch, (2 * POISON + n_pts) * 24 + n_pts * 4 + (1 << 28), f"{n} images of {rows}x{cols}")
    first = POISON * 3
    names = batch_kernels(rows, cols, n, first)
    assert ran(names, "k_labels_tma"), names

    image, near = batch_images(synth, shape, n)
    buf = torch.full((2 * POISON * 3 + n_pts * 3,), float("nan"), dtype=torch.float64, device="cuda")
    for lo in range(0, n, CHUNK):
        hi = min(n, lo + CHUNK)
        host = np.stack([image(i) for i in range(lo, hi)])
        buf[first + lo * npx * 3:first + hi * npx * 3].copy_(torch.from_numpy(host.reshape(-1)))
    del host
    labels = Guarded(torch, n_pts * 4)
    ctx = pkg.Context(rows, cols, device=0)
    try:
        ctx.set_stream(torch.cuda.current_stream().cuda_stream)
        call = lambda: ctx.extract_feature_batch_dev(buf.data_ptr() + first * 8, n, labels.ptr())  # noqa: E731
        _, delta = counted(ctx, call)
        ctx.set_stream(None)
    finally:
        ctx.close()
    del buf
    assert labels.guards_intact()
    got = labels.get(np.int32, (n, rows, cols))
    del labels
    bad = [i for i, ok in enumerate(pool_map(lambda i: np.array_equal(got[i], oracle.extract_feature(image(i))),
                                             range(n))) if not ok]
    assert not bad, (len(bad), bad[:16])
    lo, _, _ = bounds_of(near)
    assert delta >= lo, (delta, lo)


# ------------------------------------------------------------------ 2 + 3. eight sequences -------------------
SEQ_SHAPE = (64, 2048)
N_SEQ = 8
K = 32               # the bench's Fb - 1
STOPS = (1, 2, 16, 32)


def stats_frames(s):
    """the frames of sequence s whose fit totals are held to the oracle's correspondences (localize: 0.4 s each)"""
    return {s, K - 1 - s}


@pytest.fixture(scope="module")
def eight(oracle, synth):
    """Frames [K+1][N_SEQ][64][2048][3] (distinct per sequence), the pose chain (distinct per sequence) and the
    oracle walked frame by frame along it, one thread per sequence: walk[s][f] holds frame f+1's labels, nn_idx and
    nn_dist, its global cloud at the STOPS and its correspondences at stats_frames(s)."""
    r, c = SEQ_SHAPE
    frames = seq_frames(synth, SEQ_SHAPE, N_SEQ, K + 1, "small")
    pred, last, final = pose_chain(K, N_SEQ, "small")

    def walk(s):
        slam = oracle.slam(r, c, 1)
        try:
            slam.init(np.zeros(6), frames[0, s])
            out = []
            for f in range(K):
                cloud = frames[f + 1, s]
                corr = slam.localize(cloud, pred[f, s], last[f, s])[1] if f in stats_frames(s) else None
                feat, idx, dist, g = slam.frontend_frame(cloud, pred[f, s], last[f, s], final[f, s])
                out.append(SimpleNamespace(labels=feat.astype(np.int8), nn_idx=idx, nn_dist=dist, corr=corr,
                                           glob=g if f + 1 in STOPS else None))
            return out
        finally:
            slam.close()

    return SimpleNamespace(frames=frames, pred=pred, last=last, final=final, walk=pool_map(walk, range(N_SEQ)))


def frame_state(ctx, n_seq):
    """labels, nn_idx, nn_dist and global cloud of the context's last frame, [n_seq][rows][cols](...)"""
    r, c = SEQ_SHAPE
    res = ctx.frame_results_dev()
    n = n_seq * r * c
    return {"labels": dev_to_numpy(res.labels, np.int32, n).reshape(n_seq, r, c),
            "nn_idx": dev_to_numpy(res.nn_idx, np.int32, n).reshape(n_seq, r, c),
            "nn_dist": dev_to_numpy(res.nn_dist, np.float64, n).reshape(n_seq, r, c),
            "global": dev_to_numpy(res.global_, np.float64, 3 * n).reshape(n_seq, r, c, 3)}


def one_sequence(torch, eight, s):
    """sequence s alone on the device, [K+1][1][rows][cols][3]"""
    return torch.from_numpy(np.ascontiguousarray(eight.frames[:, s:s + 1])).cuda()


def assert_multi_wave(torch, n_seq):
    """one CTA per (sequence, row, 256-column tile): several resident waves per launch"""
    r, c = SEQ_SHAPE
    grid = n_seq * r * -(-c // CTA_THREADS)
    wave = resident_wave(torch)
    assert grid > wave and grid > 4 * torch.cuda.get_device_properties(0).multi_processor_count, (grid, wave)


@gpu
def test_eight_sequences_replay(pkg, eight):
    """Config 5a on one GPU: nav_frontend_sequence_dev with 8 sequences of 64x2048 side by side, one k_frame_match
    launch of 4096 CTAs per frame on a user stream (programmatic dependent launch), stopped after k = 1, 2, 16 and 32
    frames.  Each sequence's labels, nn_idx, nn_dist and global cloud equal a single-sequence replay of it (one
    k_frame_seq launch) bit for bit, and the oracle's after frame k (nn_idx / nn_dist on labelled pixels)."""
    torch = pytest.importorskip("torch")
    r, c = SEQ_SHAPE
    assert_multi_wave(torch, N_SEQ)
    need_device(torch, eight.frames.nbytes + (1 << 30), "8 sequences of 33 frames")
    d_frames = torch.from_numpy(eight.frames).cuda()
    stream = torch.cuda.Stream()
    multi = {}
    ctx = pkg.Context(r, c, device=0, n_seq=N_SEQ)
    try:
        ctx.set_stream(stream.cuda_stream)
        for k in STOPS:
            ctx.slam_init_dev(d_frames[0].data_ptr(), np.zeros((N_SEQ, 6)))
            ctx.frontend_sequence_dev(d_frames[1].data_ptr(), k, eight.pred[:k].reshape(-1, 6),
                                      eight.last[:k].reshape(-1, 6), eight.final[:k].reshape(-1, 6))
            stream.synchronize()
            multi[k] = frame_state(ctx, N_SEQ)
    finally:
        ctx.close()
    del d_frames
    for s in range(N_SEQ):
        d_one = one_sequence(torch, eight, s)
        one = pkg.Context(r, c, device=0)
        try:
            for k in STOPS:
                one.slam_init_dev(d_one[0].data_ptr(), np.zeros(6))
                one.frontend_sequence_dev(d_one[1].data_ptr(), k, eight.pred[:k, s], eight.last[:k, s],
                                          eight.final[:k, s])
                one.synchronize()
                alone = frame_state(one, 1)
                for name, a in alone.items():
                    assert a[0].tobytes() == multi[k][name][s].tobytes(), (k, s, name)
                want = eight.walk[s][k - 1]
                lab = want.labels == 1
                assert np.array_equal(multi[k]["labels"][s], want.labels), (k, s)
                assert np.array_equal(multi[k]["nn_idx"][s][lab], want.nn_idx[lab]), (k, s)
                assert multi[k]["nn_dist"][s][lab].tobytes() == want.nn_dist[lab].tobytes(), (k, s)
                assert multi[k]["global"][s].tobytes() == want.glob.tobytes(), (k, s)
        finally:
            one.close()


@gpu
def test_eight_sequences_every_frame(pkg, eight):
    """nav_frontend_sequence_out_dev with 8 sequences of 64x2048 and all four rings (the per-frame path: 4096-CTA
    k_frame_match launches, k_dedupe_stats and the fit totals over 8 x 64 x 8 partials per frame), guard bands
    intact.  Every slot of sequence s equals the slot of a single-sequence replay of it (one k_frame_seq launch in
    output mode) bit for bit; the label masks, nn_idx and nn_dist of every slot equal the oracle's, and the fit
    totals of two frames per sequence the exact sums of the oracle's correspondences (check_stats)."""
    torch = pytest.importorskip("torch")
    r, c = SEQ_SHAPE
    assert_multi_wave(torch, N_SEQ)
    need_device(torch, eight.frames.nbytes + K * N_SEQ * r * c * 13 + (1 << 30), "8 sequences with every ring")
    d_frames = torch.from_numpy(eight.frames).cuda()
    rings = Rings(torch, K, N_SEQ, r, c)
    ctx, _ = replay(pkg, torch, SEQ_SHAPE, N_SEQ, d_frames, eight.pred, eight.last, eight.final, rings,
                    rings.spec.keys())
    ctx.close()
    del d_frames
    for name in rings.spec:
        assert rings.guards_intact(name), name
    got = {name: rings.get(name) for name in rings.spec}
    del rings
    for s in range(N_SEQ):
        d_one = one_sequence(torch, eight, s)
        one = Rings(torch, K, 1, r, c)
        octx, _ = replay(pkg, torch, SEQ_SHAPE, 1, d_one, eight.pred[:, s:s + 1], eight.last[:, s:s + 1],
                         eight.final[:, s:s + 1], one, one.spec.keys())
        octx.close()
        for name in one.spec:
            assert one.guards_intact(name), (s, name)
            assert one.get(name)[:, 0].tobytes() == got[name][:, s].tobytes(), (s, name)
        del one, d_one
        mask, idx, dist, stats = (got[name][:, s] for name in ("label_mask", "nn_idx", "nn_dist", "fit_stats"))
        for f in range(K):
            want = eight.walk[s][f]
            lab = want.labels == 1
            assert np.array_equal(unpack_mask(mask[f], c), want.labels), (f, s)
            assert np.array_equal(idx[f][lab], want.nn_idx[lab]), (f, s)
            assert dist[f][lab].tobytes() == want.nn_dist[lab].tobytes(), (f, s)
            assert (idx[f][~lab] == -1).all() and (dist[f][~lab] == -1.0).all(), (f, s)
            if want.corr is not None:
                check_stats(stats[f], want.corr, SEQ_SHAPE)


# ------------------------------------------------------------------ 4. the device closed loop ----------------
@gpu
@pytest.mark.parametrize("n_seq", [8, 16])
def test_slam_run_dev_many_sequences(pkg, synth, n_seq):
    """nav_slam_run_dev with 8 and 16 sequences of 64x2048 over 6 frames, distinct starts and increments: 4096 /
    8192 clustered k_loop_step<true> CTAs per launch, the fit run by the last CTA of each sequence.  Sequence s
    equals, bit for bit, a single-sequence nav_slam_run_dev of it and nav_slam_run of it (poses, errors, totals)."""
    torch = pytest.importorskip("torch")
    shape, k = SEQ_SHAPE, 6
    assert_multi_wave(torch, n_seq)
    frames = frames_of(synth, shape, k + 1, n_seq=n_seq)
    need_device(torch, frames.nbytes + (1 << 30), f"{n_seq} sequences of {k + 1} frames")
    deltas = deltas_of(k, n_seq, seed=100 + n_seq)
    start = np.array([[3.0 * s, 0.5 * s, -0.25 * s, 0.01 * s, 0.0, 0.1 * s] for s in range(n_seq)])
    ctx, (poses, errs, stats) = dev_loop(pkg, torch, shape, frames, deltas, start)
    ctx.close()
    assert (stats[:, :, 0] > 0).all()
    for s in range(n_seq):
        one = np.ascontiguousarray(frames[:, s:s + 1])
        c1, (p1, e1, s1) = dev_loop(pkg, torch, shape, one, np.ascontiguousarray(deltas[:, s:s + 1]), start[s])
        c1.close()
        assert same_bits(poses[:, s], p1[:, 0]) and same_bits(errs[:, s], e1[:, 0]), s
        assert same_bits(stats[:, s], s1[:, 0]), s
        frames1 = np.ascontiguousarray(frames[:, s])
        with pinned(pkg, frames1):
            hctx, hp, he, hn, hs = host_loop(pkg, shape, frames1, deltas[:, s], start[s])
            hctx.close()
        assert same_bits(poses[:, s], hp) and same_bits(errs[:, s], he) and same_bits(stats[:, s], hs), s
        assert np.array_equal(stats[:, s, 0].astype(np.int64), hn), s


# ------------------------------------------------------------------ 5. large-map searches --------------------
NQ = 131072
N_ORACLE = 512   # random queries of every set held to oracle.nn_brute (2 ms per query at 1 M points, 20 at 10 M)
MAPS = ("uniform_1m", "accumulated", "uniform_10m")


def nn_problem(synth, name):
    """(points, {query set: queries}) as bench.py builds them: queries derived from every (n / 200 000)-th point of
    the uniform maps, the next frame's points in image order for the accumulated room map."""
    if name == "accumulated":
        pts, q = synth.accumulated_map(8)
        return pts, {"image_order": q}
    n = 1_000_000 if name == "uniform_1m" else 10_000_000
    pts = synth.map_points(n)
    sample = pts[::max(n // 200000, 1)]
    sets = {"jitter": synth.map_queries(sample, NQ)}
    if name == "uniform_1m":
        sets["uniform"] = synth.map_queries(sample, NQ, variant="uniform")
    return pts, {k: np.ascontiguousarray(v) for k, v in sets.items()}


def device_nn(torch, fn, d_q):
    """(idx, dist) that fn(q_ptr, nq, idx_ptr, dist_ptr, stream) leaves in buffers pre-filled with 7"""
    d_idx = torch.full((d_q.shape[0],), 7, dtype=torch.int32, device="cuda")
    d_dist = torch.full((d_q.shape[0],), 7.0, dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream()
    fn(d_q.data_ptr(), d_q.shape[0], d_idx.data_ptr(), d_dist.data_ptr(), stream.cuda_stream)
    stream.synchronize()
    return d_idx.cpu().numpy(), d_dist.cpu().numpy()


def brute_force(pkg, d_pts, tc=False):
    return lambda q, nq, i, d, s: pkg.bruteforce_nn_dev(0, d_pts.data_ptr(), d_pts.shape[0], q, nq, i, d,
                                                        use_tensor_cores=tc, stream=s)


@pytest.fixture(scope="module")
def nn_truth(pkg, oracle, synth):
    """{map: (points, query sets, {query set: (idx, dist)})}: the fp64 brute force k_bf_nn answers every query; it is
    held to oracle.nn_brute on N_ORACLE random queries of every set (a thread per block of queries)."""
    torch = pytest.importorskip("torch")
    out = {}
    for name in MAPS:
        pts, sets = nn_problem(synth, name)
        need_device(torch, pts.nbytes + (1 << 30), f"the {name} map")
        d_pts = torch.from_numpy(pts).cuda()
        truth = {}
        for qname, q in sets.items():
            idx, dist = truth[qname] = device_nn(torch, brute_force(pkg, d_pts), torch.from_numpy(q).cuda())
            assert (idx >= 0).all() and np.isfinite(dist).all(), (name, qname)
            pick = np.sort(np.random.default_rng(len(pts) + len(qname)).choice(NQ, N_ORACLE, replace=False))
            blocks = np.array_split(pick, WORKERS)
            got = pool_map(lambda b: oracle.nn_brute(pts, q[b]), blocks)
            oi, od = np.concatenate([g[0] for g in got]), np.concatenate([g[1] for g in got])
            assert_nn(idx[pick], dist[pick], oi, od, (name, qname, "fp64 brute force against the oracle"))
        del d_pts
        out[name] = (pts, sets, truth)
    return out


@gpu
@pytest.mark.parametrize("name", MAPS)
def test_kd_tree_every_query(pkg, nn_truth, name):
    """The kd tree under both split rules (nav_kdtree_build_ex on device points, nav_kdtree_nn_batch_dev on a user
    stream, as bench.py calls them; k_kd_nn_stack) answers every query of every set like the fp64 brute force."""
    torch = pytest.importorskip("torch")
    pts, sets, truth = nn_truth[name]
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_pts = torch.from_numpy(pts).cuda()
        d_sets = {qname: torch.from_numpy(q).cuda() for qname, q in sets.items()}
        for split in ("widest", "cyclic"):
            tree = pkg.KdTree(dev_ptr=d_pts.data_ptr(), n=pts.shape[0], stream=stream.cuda_stream, split=split)
            try:
                for qname, d_q in d_sets.items():
                    idx, dist = device_nn(torch, tree.nn_batch_dev, d_q)
                    assert_nn(idx, dist, *truth[qname], (name, qname, split))
            finally:
                tree.close()


@gpu
@pytest.mark.parametrize("kernel", ["plain", "conv"])
def test_stackless_kd_kernels_every_query(nn_truth, kernel):
    """NAV_KD_KERNEL=plain|conv (k_kd_nn, k_kd_nn_conv), read once per process: tests/kd_kernel_worker.py answers
    every query set of the uniform maps and the accumulated room map under both split rules, every query held to
    the fp64 brute force."""
    cases = [(name, qname) for name in ("uniform_1m", "uniform_10m") for qname in nn_truth[name][1]]
    with tempfile.TemporaryDirectory() as tmp:
        src, dst = os.path.join(tmp, "in.npz"), os.path.join(tmp, "out.npz")
        pts_a, sets_a, _ = nn_truth["accumulated"]
        arrays = {"big_pts": pts_a, "big_q": sets_a["image_order"]}
        for i, (name, qname) in enumerate(cases):
            arrays[f"pts_{i}"], arrays[f"q_{i}"] = nn_truth[name][0], nn_truth[name][1][qname]
        np.savez(src, n_cases=len(cases), **arrays)
        del arrays
        res = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "kd_kernel_worker.py"), src, dst],
                             env=dict(os.environ, NAV_KD_KERNEL=kernel), capture_output=True, text=True, timeout=900)
        assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
        got = dict(np.load(dst))
    for split in ("widest", "cyclic"):
        for i, (name, qname) in enumerate(cases):
            assert_nn(got[f"idx_{i}_{split}"], got[f"dist_{i}_{split}"], *nn_truth[name][2][qname],
                      (kernel, name, qname, split))
        assert_nn(got[f"big_idx_{split}"], got[f"big_dist_{split}"], *nn_truth["accumulated"][2]["image_order"],
                  (kernel, "accumulated", split))


@gpu
@pytest.mark.parametrize("name", ["accumulated", "uniform_1m"])
def test_tensor_cores_every_query(pkg, nn_truth, name):
    """The tensor-core brute force (bf_tc.cu: tcgen05 candidate tiles + exact binary64 re-rank) on the bench's 1 M
    maps answers every query like the fp64 brute force, and like the default kd tree -- bench.py's
    same_answers_as_kdtree, here an assertion."""
    torch = pytest.importorskip("torch")
    pts, sets, truth = nn_truth[name]
    need_device(torch, pts.nbytes + (-(-pts.shape[0] // 256)) * NQ + (1 << 30), f"tensor cores on the {name} map")
    d_pts = torch.from_numpy(pts).cuda()
    tree = pkg.KdTree(dev_ptr=d_pts.data_ptr(), n=pts.shape[0], stream=torch.cuda.current_stream().cuda_stream)
    try:
        for qname, q in sets.items():
            d_q = torch.from_numpy(q).cuda()
            ti, td = device_nn(torch, brute_force(pkg, d_pts, tc=True), d_q)
            assert_nn(ti, td, *truth[qname], (name, qname, "tensor cores against the fp64 brute force"))
            ki, kd = device_nn(torch, tree.nn_batch_dev, d_q)
            assert_nn(ti, td, ki, kd, (name, qname, "tensor cores against the kd tree"))
    finally:
        tree.close()
