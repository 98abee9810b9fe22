"""The reference tie rule (nav_set_tie_rule(ctx, NAV_TIE_REFERENCE), Context.set_tie_rule("reference")): where two
map points of a row share a query's smallest rounded distance, the blocking calls return the point the reference's
own per-row tree search returns.  Everything is compared bit for bit with the CPU oracle in tie mode 0 (the
reference-shaped trees, pinned to the reference by tests/test_golden.py), on integer-valued data full of exact and
sub-ulp ties; the per-frame count of host-resolved queries is held to the oracle's tie census."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle_lib import REF_DIR

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEP = np.array([48.0, 1.0, 0.0, 0.0, 0.0, 0.0])
UNIT = np.array([1.0, 0.0, 0.0, 0.0, 0.0, 0.0])
KTILE, KCHUNK = 256, 16  # columns per CTA tile (= one super block) and per leaf of the row map


def int_frames(rows, cols, n, seed, lo=-6, hi=7):
    """integer-valued clouds with coordinates in a few millimetres: nearly every point is an edge point, and
    equidistant map points are everywhere in a row -- in other leaves, tiles and super blocks, on both sides"""
    return np.random.default_rng(seed).integers(lo, hi, size=(n, rows, cols, 3)).astype(np.float64)


def expected_ties(oracle, cloud, pred, last, prev_global, prev_labels):
    """labelled queries whose row map is not empty and has at least two points at the smallest rounded distance"""
    feat = oracle.extract_feature(cloud)
    q = oracle.shift(oracle.transform(cloud, pred), (np.asarray(pred) - np.asarray(last))[:3])
    n = 0
    for r in range(cloud.shape[0]):
        mp = prev_global[r][prev_labels[r] == 1]
        qs = q[r][feat[r] == 1]
        if len(mp) and len(qs):
            n += int((oracle.nn_tie_count(mp, qs) >= 2).sum())
    return n


def run_frames(pkg, oracle, frames, poses, n_seq=1, depth=None, rule="reference"):
    """frontend_frame (frontend_frame_depth with depth=[distances]) over frames[1:] on a context with `rule`, per pixel
    against the oracle in tie mode 0, and the per-frame count of resolved queries against the oracle's census.
    frames: [n][n_seq][rows][cols][3]; poses[f] = (pred, last, final) per sequence.  Returns the resolved total."""
    n, rows, cols = frames.shape[0], frames.shape[2], frames.shape[3]
    ctx = pkg.Context(rows, cols, n_seq=n_seq)
    ctx.set_tie_rule(rule)
    assert ctx.tie_rule == rule
    slams = [oracle.slam(rows, cols, 0 if rule == "reference" else 1) for _ in range(n_seq)]
    start = np.zeros((n_seq, 6))
    ctx.slam_init(start, frames[0] if n_seq > 1 else frames[0, 0])
    prev = [(s.init(start[k], frames[0, k]), oracle.extract_feature(frames[0, k])) for k, s in enumerate(slams)]
    total = 0
    for f in range(1, n):
        pred, last, final = (np.asarray(p, dtype=np.float64).reshape(n_seq, 6) for p in poses[f])
        before = ctx.tie_resolve_count()
        if depth is not None:
            _, feat, idx, dist, g = ctx.frontend_frame_depth(depth[f], pred[0], last[0], final[0])
            feat, idx, dist, g = feat[None], idx[None], dist[None], g[None]
        elif n_seq > 1:
            feat, idx, dist, g = ctx.frontend_frame(frames[f], pred, last, final)
        else:
            feat, idx, dist, g = (a[None] for a in ctx.frontend_frame(frames[f, 0], pred[0], last[0], final[0]))
        want = 0
        for k, s in enumerate(slams):
            of, oi, od, og = s.frontend_frame(frames[f, k], pred[k], last[k], final[k])
            assert np.array_equal(feat[k], of), (f, k, "labels")
            bad = np.argwhere(idx[k] != oi)
            assert bad.size == 0, (f, k, "nn_idx", bad[:5].tolist(), idx[k][tuple(bad[0])], oi[tuple(bad[0])])
            assert np.array_equal(dist[k], od), (f, k, "nn_dist")
            assert np.array_equal(g[k], og), (f, k, "mapped cloud")
            want += expected_ties(oracle, frames[f, k], pred[k], last[k], *prev[k])
            prev[k] = (og, of)
        got = ctx.tie_resolve_count() - before
        assert got == (want if rule == "reference" else 0), (f, got, want)
        total += got
    for s in slams:
        s.close()
    ctx.close()
    return total


def walk(n, step=UNIT):
    """poses of a straight walk: prediction = last + step, final = prediction (integer, no rotation: exact)"""
    out, last = [None], np.zeros(6)
    for _ in range(1, n):
        pred = last + step
        out.append((pred, last, pred))
        last = pred
    return out


# name -> (frames [n][n_seq][rows][cols][3], poses, n_seq)
def _case(name, synth):
    if name == "l9_16x1800":
        fr = synth.l9_sequence(4)[:, None]
        return fr, walk(4, STEP), 1
    if name == "int_4x2048":
        return int_frames(4, 2048, 4, seed=1)[:, None], walk(4), 1
    if name == "int_3x4100_superbox":
        return int_frames(3, 4100, 3, seed=2)[:, None], walk(3), 1
    if name == "int_1x17":
        return int_frames(1, 17, 5, seed=3, lo=-2, hi=3)[:, None], walk(5), 1
    if name == "int_5x33":
        return int_frames(5, 33, 5, seed=4, lo=-3, hi=4)[:, None], walk(5), 1
    if name == "empty_rows":
        fr = int_frames(4, 600, 4, seed=5)
        fr[:, 1] = 0.0   # no edge points in any frame: no map, no query
        fr[0, 2] = 0.0   # an empty map under labelled queries
        return fr[:, None], walk(4), 1
    if name == "duplicate_xyz":
        fr = int_frames(4, 700, 4, seed=6)
        fr[:, :, 300:332] = fr[:, :, 20:52]     # the same xyz in other leaves and tiles of the row
        fr[:, :, 600:616] = fr[:, :, 40:56]
        return fr[:, None], walk(4), 1
    if name == "sub_ulp_1e9":
        # queries 1e9 mm from their row map (pos_last is 1e9 mm ahead of the pose the map was built with): every
        # dsq is about 1e18, binary64 holds it to 128, and the rounded distances of map points whose (dy^2 + dz^2)
        # differ by a few hundred are equal -- sqrt ties between different squared distances, all over the row
        fr = int_frames(4, 2048, 4, seed=7)[:, None]
        poses, last = [None], np.zeros(6)
        for _ in range(1, 4):
            far = last + np.array([1e9, 0, 0, 0, 0, 0])
            pred = far + UNIT
            poses.append((pred, far, last + UNIT))
            last = last + UNIT
        return fr, poses, 1
    if name == "n_seq2":
        fr = np.stack([int_frames(3, 600, 4, seed=8), int_frames(3, 600, 4, seed=9)], axis=1)
        poses = [None] + [(np.stack([p[0], p[0] + UNIT]), np.stack([p[1], p[1] + UNIT]), np.stack([p[2], p[2] + UNIT]))
                          for p in walk(4)[1:]]
        return fr, poses, 2
    raise KeyError(name)


CASES = ["l9_16x1800", "int_4x2048", "int_3x4100_superbox", "int_1x17", "int_5x33", "empty_rows", "duplicate_xyz",
         "sub_ulp_1e9", "n_seq2"]


@pytest.mark.parametrize("name", CASES)
def test_frontend_frame_matches_the_reference_oracle(pkg, oracle, synth, name):
    frames, poses, n_seq = _case(name, synth)
    assert run_frames(pkg, oracle, frames, poses, n_seq=n_seq) > 0


def test_constructed_ties_span_leaves_tiles_and_both_sides(oracle):
    """the integer 4x2048 frames put tied map points in other leaves and other tiles (= super blocks) of the row than
    the query's seed, below and above it -- the cases the pruning argument of search_row covers"""
    fr = int_frames(4, 2048, 4, seed=1)
    g0 = fr[0]  # identity pose: the map is the cloud itself
    lab0 = oracle.extract_feature(fr[0])
    q = oracle.shift(oracle.transform(fr[1], UNIT), UNIT[:3])
    lab1 = oracle.extract_feature(fr[1])
    seen = {"other_leaf": 0, "other_tile_below": 0, "other_tile_above": 0}
    for r in range(4):
        cols = np.flatnonzero(lab0[r] == 1)
        mp = g0[r][cols]
        for qc in np.flatnonzero(lab1[r] == 1)[::7]:
            d = np.sqrt(((mp - q[r, qc]) ** 2).sum(axis=1))
            tied = cols[d == d.min()]
            if len(tied) < 2:
                continue
            seen["other_leaf"] += int(np.any(tied // KCHUNK != qc // KCHUNK))
            seen["other_tile_below"] += int(np.any(tied // KTILE < qc // KTILE))
            seen["other_tile_above"] += int(np.any(tied // KTILE > qc // KTILE))
    assert all(v > 0 for v in seen.values()), seen


def test_depth_input_matches_the_reference_oracle(pkg, oracle):
    rows, cols = 8, 300
    rng = np.random.default_rng(10)
    depth = rng.integers(1000, 1006, size=(4, rows, cols)).astype(np.int32)
    frames = np.stack([oracle.convert(d) for d in depth])[:, None]
    run_frames(pkg, oracle, frames, walk(4), depth=depth)


def test_room_data_has_no_ties(pkg, oracle, synth):
    """fp64 room data (64x2048): nothing is flagged, and the outputs are the reference's"""
    frames = synth.room_sequence(64, 2048, 3)[:, None]
    assert run_frames(pkg, oracle, frames, walk(3, STEP)) == 0


def test_default_rule_is_untouched(pkg, oracle):
    """a fresh context and one switched to "reference" and back give the same lowest-index answers on tied data (the
    oracle's tie mode 1), and resolve nothing"""
    frames = int_frames(4, 2048, 4, seed=1)[:, None]
    assert run_frames(pkg, oracle, frames, walk(4), rule="lowest_index") == 0
    a = pkg.Context(4, 2048)
    b = pkg.Context(4, 2048)
    b.set_tie_rule("reference")
    b.set_tie_rule("lowest_index")
    assert a.tie_rule == b.tie_rule == "lowest_index"
    for ctx in (a, b):
        ctx.slam_init(np.zeros(6), frames[0, 0])
    for f, (pred, last, final) in enumerate(walk(4)[1:], start=1):
        ra, rb = a.frontend_frame(frames[f, 0], pred, last, final), b.frontend_frame(frames[f, 0], pred, last, final)
        for x, y in zip(ra, rb):
            assert np.array_equal(x, y)
    assert a.tie_resolve_count() == b.tie_resolve_count() == 0
    with pytest.raises(ValueError):
        a.set_tie_rule("first_visited")
    assert a.L.nav_set_tie_rule(a.h, 2) != 0 and b"tie rule" in a.L.nav_last_error()
    a.close()
    b.close()


def _golden_16x1800(pkg, synth):
    """frames 1-2 of the reference-generated tests/golden/ref_16x1800.npz, exactly: poses, errors, global clouds"""
    import hashlib
    g = np.load(os.path.join(ROOT, "tests", "golden", "ref_16x1800.npz"))
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()  # noqa: E731
    clouds = [synth.room_frame(16, 1800, f, cfg=2, elev=(-15, 15), integer_mm=True) for f in range(3)]
    ctx = pkg.Context(16, 1800)
    ctx.set_tie_rule("reference")
    assert sha(ctx.slam_init(np.zeros(6), clouds[0])) == g["global_sha256"][0]
    last = np.zeros(6)
    for f in (1, 2):
        p, err = ctx.slam_localization(clouds[f], last + STEP, last)
        assert np.array_equal(p, g["poses"][f]), (f, p - g["poses"][f])
        assert err == g["errors"][f]
        assert sha(ctx.slam_mapping(p, clouds[f])) == g["global_sha256"][f]
        last = p
    assert ctx.tie_resolve_count() > 0
    ctx.close()


def test_whole_step_is_the_reference_bit_for_bit(pkg, oracle, synth):
    """slam_match + slam_localization + slam_mapping chained over 10 integer-mm 16x1800 frames: correspondence lists,
    poses, errors and mapped clouds equal to the oracle in tie mode 0; frames 1-2 equal to the reference's own
    golden vectors (where the lowest-index rule can only hold the pose to 5e-3)"""
    frames = synth.l9_sequence(11)
    ctx = pkg.Context(16, 1800)
    ctx.set_tie_rule("reference")
    slam = oracle.slam(16, 1800, 0)
    pos = np.zeros(6)
    assert np.array_equal(ctx.slam_init(pos, frames[0]), slam.init(pos, frames[0]))
    last = pos
    for f in range(1, 11):
        pred = last + STEP
        corr = ctx.slam_match(frames[f], pred, last)
        p_or, corr_or, err_or, _ = slam.localize(frames[f], pred, last)
        assert np.array_equal(corr, corr_or), f
        p, err = ctx.slam_localization(frames[f], pred, last)
        assert np.array_equal(p, p_or), (f, p - p_or)
        assert err == err_or
        assert np.array_equal(ctx.slam_mapping(p, frames[f]), slam.map(p_or, frames[f])), f
        last = p
    assert ctx.tie_resolve_count() > 0
    slam.close()
    ctx.close()
    _golden_16x1800(pkg, synth)


def test_refused_calls_leave_the_context_usable(pkg, oracle):
    import torch
    rows, cols = 4, 600
    frames = int_frames(rows, cols, 3, seed=11)
    ctx = pkg.Context(rows, cols)
    ctx.set_tie_rule("reference")
    slam = oracle.slam(rows, cols, 0)
    ctx.slam_init(np.zeros(6), frames[0])
    slam.init(np.zeros(6), frames[0])
    L = ctx.L
    pred, last, final = walk(2)[1]
    nbytes = frames[1].nbytes
    h_mem = L.nav_host_alloc(nbytes * 4)
    h = np.ctypeslib.as_array(C.cast(h_mem, C.POINTER(C.c_double)), shape=(4,) + frames[1].shape)
    h[0] = frames[1]
    hp = [h_mem + k * nbytes for k in range(4)]
    d = torch.from_numpy(frames[1:3].copy()).cuda()
    d_idx = torch.zeros(2 * rows * cols, dtype=torch.int32, device="cuda")
    ctx.slam_prefetch(cloud_ptr=hp[0])  # allowed: it only uploads and labels, its consumer refuses
    refused = {
        "nav_frontend_frame_dev": lambda: ctx.frontend_frame_dev(d.data_ptr(), pred, last, final),
        "nav_frontend_sequence_dev": lambda: ctx.frontend_sequence_dev(d.data_ptr(), 2, np.stack([pred, pred]),
                                                                       np.stack([last, last]), np.stack([final, final])),
        "nav_frontend_sequence_out_dev": lambda: ctx.frontend_sequence_out_dev(
            d.data_ptr(), 2, np.stack([pred, pred]), np.stack([last, last]), np.stack([final, final]),
            nn_idx=d_idx.data_ptr()),
        "nav_frontend_frame_async": lambda: ctx.frontend_frame_async(hp[0], pred, last, final, hp[1], None, None, None),
        "nav_frontend_submit": lambda: ctx.frontend_submit(pred, last, final, cloud=hp[0], global_out=hp[1]),
        "nav_slam_localization_fast": lambda: ctx.slam_localization_fast(frames[1], pred, last),
        "nav_slam_run": lambda: ctx.slam_run([hp[0]], UNIT[None], np.zeros(6)),
    }
    for name, call in refused.items():
        before = ctx.launch_count()
        with pytest.raises(pkg.NavError, match="tie rule") as e:
            call()
        assert name in str(e.value)
        assert ctx.launch_count() == before, name
    from importlib import import_module
    NavPos = import_module("nav-slam_b200.binding").NavPos
    P = lambda v: C.byref(NavPos(*[float(x) for x in v]))  # noqa: E731
    L.nav_frontend_frame_depth_async.restype = C.c_int
    before = ctx.launch_count()
    assert L.nav_frontend_frame_depth_async(ctx.h, hp[2], P(pred), P(last), P(final), None, None, None, None, None) != 0
    assert b"tie rule" in L.nav_last_error() and ctx.launch_count() == before
    torch.cuda.synchronize()
    # the context still runs a supported call exactly as if nothing had been asked of it
    feat, idx, dist, g = ctx.frontend_frame(frames[1], pred, last, final)
    of, oi, od, og = slam.frontend_frame(frames[1], pred, last, final)
    assert np.array_equal(feat, of) and np.array_equal(idx, oi) and np.array_equal(dist, od) and np.array_equal(g, og)
    L.nav_host_free(h_mem)
    slam.close()
    ctx.close()


SHIM_RUN = r'''
import importlib, json, sys, os, hashlib
import numpy as np
sys.path.insert(0, %r)
nav = importlib.import_module("nav-slam_b200")
sb = importlib.import_module("nav-slam_b200.shim_binding")
frames = nav.synth.l9_sequence(5)
shim = sb.ShimSlam(16, 1800)
pc = shim.pack_cloud(frames[0], ts=0)
fd = os.dup(1); os.dup2(os.open(os.devnull, os.O_WRONLY), 1)
shim.init_slam(np.zeros(6), pc)
last = np.zeros(6); out = []
for f in range(1, 5):
    pc[8:] = frames[f].reshape(-1).view(np.uint8)
    p = shim.slam_localization(pc, last + np.array([48.0, 1.0, 0, 0, 0, 0]), last)
    shim.slam_mapping(p, pc)
    out.append({"pose": [float(v).hex() for v in p], "error": float(shim.error).hex(),
                "global": hashlib.sha256(shim.global_cloud(f).tobytes()).hexdigest()})
    last = p
g0 = hashlib.sha256(shim.global_cloud(0).tobytes()).hexdigest()
os.dup2(fd, 1)
print(json.dumps({"frames": out, "global0": g0}))
shim.release()
''' % ROOT


def _shim_env(**kv):
    e = {k: v for k, v in os.environ.items() if not k.startswith("NAVSLAM_")}
    e.update(kv)
    return e


def test_shim_reference_ties_match_the_oracle(oracle, synth):
    """NAVSLAM_TIES=reference: init_slam / slam_localization / slam_mapping on 16x1800 L9 frames give the oracle's tie
    mode 0 bit for bit (poses, attr->error, global clouds).  The switch is read once per process: a process of its own."""
    import hashlib
    res = subprocess.run([sys.executable, "-c", SHIM_RUN], env=_shim_env(NAVSLAM_TIES="reference"), capture_output=True,
                         text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    got = json.loads(res.stdout.strip().splitlines()[-1])
    frames = synth.l9_sequence(5)
    slam = oracle.slam(16, 1800, 0)
    assert got["global0"] == hashlib.sha256(slam.init(np.zeros(6), frames[0]).tobytes()).hexdigest()
    last = np.zeros(6)
    for f in range(1, 5):
        p, _, err, _ = slam.localize(frames[f], last + STEP, last)
        g = slam.map(p, frames[f])
        want = {"pose": [float(v).hex() for v in p], "error": float(err).hex(),
                "global": hashlib.sha256(g.tobytes()).hexdigest()}
        assert got["frames"][f - 1] == want, f
        last = p
    slam.close()


def test_shim_refuses_reference_ties_with_the_stats_fit():
    res = subprocess.run([sys.executable, "-c", SHIM_RUN], env=_shim_env(NAVSLAM_TIES="reference", NAVSLAM_ADAM="stats"),
                         capture_output=True, text=True, timeout=600)
    assert res.returncode != 0
    assert "NAVSLAM_ADAM=stats cannot be combined with NAVSLAM_TIES=reference" in res.stderr


def test_unmodified_main_l9_config2_byte_identical(synth, tmp_path):
    """BASELINE config 2 with NAVSLAM_TIES=reference: the reference's unmodified L9 main linked against the shim writes
    the reference program's CSV and stdout byte for byte"""
    ref_exe = os.path.join(REF_DIR, "navref_l9_16x1800")
    shim_exe = os.path.join(REF_DIR, "navshim_l9_16x1800")
    if not (os.path.exists(ref_exe) and os.path.exists(shim_exe)):
        pytest.skip("reference mains not built (needs /root/reference at build time)")
    csv_in = synth.l9_csv(synth.l9_sequence(4))
    outs = []
    for exe, sub, env in ((ref_exe, "ref", os.environ.copy()), (shim_exe, "shim", _shim_env(NAVSLAM_TIES="reference"))):
        wd = tmp_path / sub
        wd.mkdir()
        (wd / "parsed_data.csv").write_text(csv_in)
        res = subprocess.run([exe], cwd=str(wd), env=env, capture_output=True, timeout=600)
        assert res.returncode == 0, res.stderr.decode(errors="replace")[-2000:]
        outs.append((res.stdout, (wd / "point_cloud_data.csv").read_bytes()))
    assert outs[1][1] == outs[0][1]
    assert outs[1][0] == outs[0][0]
