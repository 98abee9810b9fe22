"""Integer-millimetre input (the reference's L9 sensor, src/main.c:77-128): frames cross PCIe as int32 [n][3] and are
widened on the device.  Every int32 is exact in binary64, so every output must equal, bit for bit, the xyz call on
mm.astype(np.float64).  The CPU tests hold the int32 L9 reader and to_mm() to the double reader and to one
acceptance rule; the GPU tests compare each mm entry point with its xyz twin.

The int32 frames are made with np.rint(x).astype(np.int32), not to_mm(): np.rint keeps the sign of a zero, and the
synthetic L9 data holds -0.0 (which the CSV writes as "0"), so to_mm() refuses it."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

STEP = np.array([48.0, 1.0, 0.0, 0.0, 0.0, 0.0])
UNIT = np.array([1.0, 0.0, 0.0, 0.0, 0.0, 0.0])
I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1


def bits(a):
    return np.ascontiguousarray(a).tobytes()


def same(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and bits(a) == bits(b)


def _write(tmp_path, text, name="parsed_data.csv"):
    p = os.path.join(str(tmp_path), name)
    with open(p, "w", newline="") as f:
        f.write(text)
    return p


# ------------------------------------------------------------------------------------------------- CPU -----------
def test_every_exported_function_with_arguments_has_argtypes(pkg):
    """without argtypes ctypes passes Python ints as 32-bit C ints: a 64-bit buffer address is cut short"""
    hdr = open(os.path.join(ROOT, "include", "navslam_b200.h")).read()
    params = dict(re.findall(r"\b(nav_[a-z0-9_]+)\s*\(([^)]*)\)", hdr))
    L = pkg.load_library()
    missing = [s for s in pkg.binding.EXPORTS if params[s].strip() not in ("", "void") and getattr(L, s).argtypes is None]
    assert not missing, missing


READ_MM_FIRST = r"""
import importlib, sys
import numpy as np
sys.path.insert(0, %r)
nav = importlib.import_module("nav-slam_b200")
mm, ts = nav.l9_csv_read_mm(sys.argv[1], 16, 1800, 10)   # the first library call of the process
print(mm.shape, int(np.abs(mm).sum()), [int(t) for t in ts])
"""


def test_reader_mm_as_the_first_call_of_a_process(pkg, synth, tmp_path):
    """a fresh process: the 3.5 MB frame buffer is mmapped far above 2 GiB, where a truncated pointer would crash"""
    x = synth.l9_sequence(3)
    path = _write(tmp_path, synth.l9_csv(x))
    r = subprocess.run([sys.executable, "-c", READ_MM_FIRST % ROOT, path], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == f"(3, 16, 1800, 3) {int(np.abs(np.rint(x)).sum())} [0, 1, 2]"


def test_reader_mm_widens_to_the_double_reader(pkg, synth, tmp_path):
    path = _write(tmp_path, synth.l9_csv(synth.l9_sequence(3)))
    frames, ts = pkg.l9_csv_read(path, 16, 1800, 10)
    mm, ts_mm = pkg.l9_csv_read_mm(path, 16, 1800, 10)
    assert len(frames) == len(mm) == 3 and mm.dtype == np.int32
    assert np.array_equal(ts, ts_mm) and list(ts) == [0, 1, 2]
    assert same(mm.astype(np.float64), frames)


def test_reader_mm_skips_out_of_image_records_and_overflows_like_the_double_reader(pkg, tmp_path):
    rows, cols = 3, 5
    lines = ["frame,row,col,x,y,z,conf"]
    rng = np.random.default_rng(5)
    for f in (7, 9, 12):
        for _ in range(20):
            r, c = int(rng.integers(-1, rows + 1)), int(rng.integers(-2, cols + 2))  # some outside the image
            x, y, z = (int(v) for v in rng.integers(-5000, 5000, 3))
            lines.append(f"{f},{r},{c},{x},{y},{z},100")
    path = _write(tmp_path, "\n".join(lines) + "\n")
    frames, ts = pkg.l9_csv_read(path, rows, cols, 3)
    mm, ts_mm = pkg.l9_csv_read_mm(path, rows, cols, 3)
    assert np.array_equal(ts, ts_mm) and len(mm) == len(frames) == 3
    assert same(mm.astype(np.float64), frames)
    for read in (pkg.l9_csv_read, pkg.l9_csv_read_mm):  # one frame more than there is room for
        with pytest.raises(pkg.NavError, match="more than 2 frames"):
            read(path, rows, cols, 2)


ACCEPTED = {"1e3": 1000, "+7": 7, "0012": 12, "-2147483648": I32_MIN, "2147483647": I32_MAX}
REJECTED = ["12.5", "-0", "2147483648", "1e10", "nan", "inf"]


def test_reader_mm_accepts_exact_integers_in_any_syntax(pkg, tmp_path):
    text = "frame,row,col,x,y,z,conf\n" + "".join(f"0,0,{c},{v},{v},{v},1\n" for c, v in enumerate(ACCEPTED))
    path = _write(tmp_path, text)
    mm, _ = pkg.l9_csv_read_mm(path, 1, len(ACCEPTED), 2)
    frames, _ = pkg.l9_csv_read(path, 1, len(ACCEPTED), 2)
    assert mm[0, 0].tolist() == [[v] * 3 for v in ACCEPTED.values()]
    assert same(mm.astype(np.float64), frames)


@pytest.mark.parametrize("value", REJECTED)
@pytest.mark.parametrize("axis", [0, 2])
def test_reader_mm_rejects_inexact_values_naming_line_and_value(pkg, tmp_path, value, axis):
    xyz = ["1", "2", "3"]
    xyz[axis] = value
    text = "frame,row,col,x,y,z,conf\n0,0,0,4,5,6,1\n0,0,1,7,8,9,1\n" + f"0,0,2,{','.join(xyz)},1\n"
    path = _write(tmp_path, text)
    pkg.l9_csv_read(path, 1, 3, 2)  # the double reader takes it
    with pytest.raises(pkg.NavError) as e:
        pkg.l9_csv_read_mm(path, 1, 3, 2)
    msg = str(e.value)
    assert "nav_l9_csv_read_mm" in msg and "line 4 " in msg and f"'{value}'" in msg and f"{'xyz'[axis]} =" in msg


def test_to_mm_follows_the_reader_rule(pkg):
    vals = np.array([float(v) for v in ACCEPTED], dtype=np.float64)
    assert list(pkg.to_mm(np.stack([vals, vals, vals], axis=-1))[:, 0]) == list(ACCEPTED.values())
    for v in REJECTED:
        a = np.zeros((2, 3))
        a[1, 1] = float(v)
        with pytest.raises(ValueError, match=r"index \(1, 1\)"):
            pkg.to_mm(a)
    x = np.rint(np.random.default_rng(1).uniform(-1e5, 1e5, (4, 7, 3))) + 0.0  # + 0.0 turns -0.0 into +0.0
    assert same(pkg.to_mm(x).astype(np.float64), x)


def test_to_mm_refuses_the_negative_zeros_of_synthetic_l9_data(pkg, synth):
    x = synth.l9_sequence(1)
    assert np.any((x == 0) & np.signbit(x))
    with pytest.raises(ValueError, match="-0.0"):
        pkg.to_mm(x)
    m = np.rint(x).astype(np.int32)  # what the GPU tests feed: the zeros come back as +0.0
    assert np.array_equal(m.astype(np.float64), x)


# ------------------------------------------------------------------------------------------------- GPU -----------
def mm_frames(x):
    """int32 frames and the float64 clouds they stand for"""
    m = np.ascontiguousarray(np.rint(x).astype(np.int32))
    return m, m.astype(np.float64)


def walk(n, step=UNIT, n_seq=1):
    out, last = [None], np.zeros((n_seq, 6))
    for _ in range(1, n):
        pred = last + step
        out.append((pred, last, pred))
        last = pred
    return out


def _frame_case(name, synth):
    """-> (int32 frames [n][n_seq][rows][cols][3], n_seq, step)"""
    rng = np.random.default_rng(100 + FRAME_CASES.index(name))
    if name == "l9_16x1800":
        return mm_frames(synth.l9_sequence(4)[:, None])[0], 1, STEP
    if name == "room_64x2048":
        return mm_frames(synth.room_sequence(64, 2048, 3, integer_mm=True)[:, None])[0], 1, STEP
    if name == "1x17":
        return rng.integers(-40, 40, (5, 1, 1, 17, 3)).astype(np.int32), 1, UNIT
    if name == "3x4100":
        return rng.integers(-3000, 3000, (3, 1, 3, 4100, 3)).astype(np.int32), 1, UNIT
    if name == "5x33_nseq2":
        return rng.integers(-300, 300, (4, 2, 5, 33, 3)).astype(np.int32), 2, UNIT
    if name == "extremes_6x96":
        m = rng.integers(-2000, 2000, (4, 1, 6, 96, 3)).astype(np.int64)
        m[:, :, :, ::7] = 0                                    # invalid returns (0,0,0)
        m[:, :, 1, 10:30, 0] = I32_MAX                         # points at the ends of the int32 range
        m[:, :, 2, 40:60] = I32_MIN
        m[:, :, 3, 5:90:3, 1] = rng.choice([I32_MIN, I32_MAX], size=(4, 1, 29))
        return m.astype(np.int32), 1, UNIT
    raise KeyError(name)


FRAME_CASES = ["l9_16x1800", "room_64x2048", "1x17", "3x4100", "5x33_nseq2", "extremes_6x96"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", FRAME_CASES)
def test_frontend_frame_mm_equals_the_xyz_call(pkg, synth, name):
    mm, n_seq, step = _frame_case(name, synth)
    xyz = mm.astype(np.float64)
    n, rows, cols = mm.shape[0], mm.shape[2], mm.shape[3]
    sq = (lambda a: a[:, 0]) if n_seq == 1 else (lambda a: a)
    a, b = pkg.Context(rows, cols, n_seq=n_seq), pkg.Context(rows, cols, n_seq=n_seq)
    start = np.zeros((n_seq, 6))
    for ctx in (a, b):
        ctx.slam_init(start, sq(xyz[:1])[0])
    for f, (pred, last, final) in enumerate(walk(n, step, n_seq)[1:], start=1):
        launches = b.launch_count()
        want = a.frontend_frame(sq(xyz[f:f + 1])[0], pred, last, final)
        got = b.frontend_frame_mm(sq(mm[f:f + 1])[0], pred, last, final)
        assert b.launch_count() == launches + 2  # the widening, then the frame kernel
        for w, g, what in zip(want, got, ("labels", "nn_idx", "nn_dist", "global")):
            assert same(w, g), (f, what)
    a.close()
    b.close()


@pytest.mark.gpu
def test_frontend_frame_mm_under_the_reference_tie_rule(pkg, oracle, synth):
    mm, _, _ = _frame_case("l9_16x1800", synth)
    xyz = mm.astype(np.float64)
    a, b = pkg.Context(16, 1800), pkg.Context(16, 1800)
    slam = oracle.slam(16, 1800, 0)
    for ctx in (a, b):
        ctx.set_tie_rule("reference")
        ctx.slam_init(np.zeros(6), xyz[0, 0])
    slam.init(np.zeros(6), xyz[0, 0])
    for f, (pred, last, final) in enumerate(walk(4, STEP)[1:], start=1):
        pred, last, final = pred[0], last[0], final[0]
        got = b.frontend_frame_mm(mm[f, 0], pred, last, final)
        a.frontend_frame(xyz[f, 0], pred, last, final)
        want = slam.frontend_frame(xyz[f, 0], pred, last, final)
        for w, g, what in zip(want, got, ("labels", "nn_idx", "nn_dist", "global")):
            assert np.array_equal(w, g), (f, what)
        assert b.tie_resolve_count() == a.tie_resolve_count(), f
    assert b.tie_resolve_count() > 0
    slam.close()
    a.close()
    b.close()


def _pinned(arr):
    import torch
    return torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(16, 1800, 1), (5, 33, 2)])
def test_submit_mm_pipelined_equals_submit_with_the_cloud(pkg, synth, shape):
    import torch
    rows, cols, n_seq = shape
    n = 8
    if n_seq == 1:
        mm = mm_frames(synth.room_sequence(rows, cols, n, cfg=2, elev=(-15.0, 15.0), integer_mm=True))[0]
        step = STEP
    else:
        mm = np.random.default_rng(3).integers(-300, 300, (n, n_seq, rows, cols, 3)).astype(np.int32)
        step = UNIT
    xyz = mm.astype(np.float64)
    h_mm, h_xyz = _pinned(mm), _pinned(xyz)
    nch = (cols + 15) // 16
    res = []
    for kind in ("xyz", "mm"):
        ctx = pkg.Context(rows, cols, n_seq=n_seq)
        ctx.slam_init(np.zeros((n_seq, 6)), xyz[0])
        out = {k: torch.zeros((n,) + s, dtype=t).pin_memory() for k, s, t in (
            ("mask", (n_seq, rows, nch), torch.int32), ("idx", (n_seq, rows, cols), torch.int32),
            ("dist", (n_seq, rows, cols), torch.float64), ("glob", (n_seq, rows, cols, 3), torch.float64))}
        for f, (pred, last, final) in enumerate(walk(n, step, n_seq)[1:], start=1):
            kw = dict(mask_out=out["mask"][f].data_ptr(), nn_idx_out=out["idx"][f].data_ptr(),
                      nn_dist_out=out["dist"][f].data_ptr(), global_out=out["glob"][f].data_ptr())
            if kind == "xyz":
                ctx.frontend_submit(pred, last, final, cloud=h_xyz[f].data_ptr(), **kw)
            else:
                ctx.frontend_submit_mm(h_mm[f].data_ptr(), pred, last, final, **kw)
        ctx.frontend_wait()
        res.append({k: v.numpy().copy() for k, v in out.items()})
        ctx.close()
    for k in res[0]:
        assert same(res[0][k], res[1][k]), k
    assert (res[1]["mask"][1:] != 0).any() and (res[1]["idx"][1:] >= 0).any()


@pytest.mark.gpu
def test_interleaved_xyz_mm_and_depth_submissions_equal_blocking_calls(pkg, synth):
    rows, cols, n = 16, 1800, 7
    x = synth.room_sequence(rows, cols, n, cfg=2, elev=(-15.0, 15.0), integer_mm=True)
    mm, xyz = mm_frames(x)
    depth = np.clip(np.rint(np.linalg.norm(xyz, axis=-1)), 1, 60000).astype(np.int32)
    h_mm, h_xyz, h_depth = _pinned(mm), _pinned(xyz), _pinned(depth)
    import torch
    feat = torch.zeros((n, rows, cols), dtype=torch.int32).pin_memory()
    idx = torch.zeros((n, rows, cols), dtype=torch.int32).pin_memory()
    dist = torch.zeros((n, rows, cols), dtype=torch.float64).pin_memory()
    glob = torch.zeros((n, rows, cols, 3), dtype=torch.float64).pin_memory()
    a, b = pkg.Context(rows, cols), pkg.Context(rows, cols)
    for ctx in (a, b):
        ctx.slam_init(np.zeros(6), xyz[0])
    kinds = ["xyz", "mm", "depth", "mm", "xyz", "depth"]
    want = {}
    for f, ((pred, last, final), kind) in enumerate(zip(walk(n, STEP)[1:], kinds), start=1):
        pred, last, final = pred[0], last[0], final[0]
        kw = dict(feature_out=feat[f].data_ptr(), nn_idx_out=idx[f].data_ptr(), nn_dist_out=dist[f].data_ptr(),
                  global_out=glob[f].data_ptr())
        if kind == "xyz":
            b.frontend_submit(pred, last, final, cloud=h_xyz[f].data_ptr(), **kw)
            want[f] = a.frontend_frame(xyz[f], pred, last, final)
        elif kind == "mm":
            b.frontend_submit_mm(h_mm[f].data_ptr(), pred, last, final, **kw)
            want[f] = a.frontend_frame_mm(mm[f], pred, last, final)
        else:
            b.frontend_submit(pred, last, final, distances=h_depth[f].data_ptr(), **kw)
            want[f] = a.frontend_frame_depth(depth[f], pred, last, final)[1:]
    b.frontend_wait()
    for f, w in want.items():
        got = (feat[f].numpy(), idx[f].numpy(), dist[f].numpy(), glob[f].numpy())
        for wv, gv, what in zip(w, got, ("labels", "nn_idx", "nn_dist", "global")):
            assert same(np.ascontiguousarray(wv), np.ascontiguousarray(gv)), (f, kinds[f - 1], what)
    a.close()
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(16, 1800), (2, 4100)])  # one k_loop_step launch per frame / three launches
def test_slam_run_mm_equals_slam_run_xyz(pkg, synth, shape):
    rows, cols = shape
    n = 9
    mm, xyz = mm_frames(synth.room_sequence(rows, cols, n, cfg=2, elev=(-15.0, 15.0), integer_mm=True))
    h_mm, h_xyz = _pinned(mm), _pinned(xyz)
    steps = np.tile(STEP + np.array([-2.0, 0.5, 0, 0, 0, 0]), (n - 1, 1))
    out = []
    for kind in ("xyz", "mm"):
        ctx = pkg.Context(rows, cols)
        ctx.slam_init(np.zeros(6), xyz[0])
        src = h_mm if kind == "mm" else h_xyz
        out.append(ctx.slam_run([src[f].data_ptr() for f in range(1, n)], steps, np.zeros(6), mm_input=kind == "mm")
                   + (ctx.slam_fit_stats(),))
        if kind == "mm":
            with pytest.raises(ValueError, match="exclude"):
                ctx.slam_run([h_mm[1].data_ptr()], steps[:1], np.zeros(6), depth_input=True, mm_input=True)
        ctx.close()
    (pa, ea, na, sa), (pb, eb, nb, sb) = out
    assert same(pa, pb) and same(ea, eb) and same(na, nb) and same(sa, sb)
    assert (nb > 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["mm", "mixed"])
def test_prefetch_mm_chain_equals_the_xyz_chain(pkg, synth, mode):
    rows, cols, n = 16, 1800, 8
    mm, xyz = mm_frames(synth.l9_sequence(n))
    h_mm, h_xyz = _pinned(mm), _pinned(xyz)
    step = STEP + np.array([-2.0, 0.5, 0, 0, 0, 0])
    runs = []
    for kind in ("xyz", mode):
        ctx = pkg.Context(rows, cols)
        ctx.slam_init(np.zeros(6), xyz[0])

        def prefetch(f):
            use_mm = kind == "mm" or (kind == "mixed" and f % 2 == 1)  # mixed: xyz and mm slots alternate
            if use_mm:
                ctx.slam_prefetch(mm_ptr=h_mm[f].data_ptr())
            else:
                ctx.slam_prefetch(cloud_ptr=h_xyz[f].data_ptr())

        prefetch(1)
        prefetch(2)
        last, rec = np.zeros(6), []
        for f in range(1, n):
            if f + 2 < n:
                prefetch(f + 2)
            p, err, nc = ctx.slam_localization_fast_ptr(None, last + step, last)
            rec.append((p, err, nc, ctx.slam_fit_stats(), ctx.slam_mapping(p, None)))
            last = p
        runs.append(rec)
        ctx.close()
    for f, (ra, rb) in enumerate(zip(*runs), start=1):
        assert same(ra[0], rb[0]) and ra[1] == rb[1] and ra[2] == rb[2], f
        assert same(ra[3], rb[3]) and same(ra[4], rb[4]), f


@pytest.mark.gpu
def test_refusals_name_the_call_and_queue_nothing(pkg, oracle):
    import torch
    rows, cols = 4, 600
    mm = np.random.default_rng(11).integers(-6, 7, (3, rows, cols, 3)).astype(np.int32)
    xyz = mm.astype(np.float64)
    h_mm, h_xyz = _pinned(mm), _pinned(xyz)
    out = torch.zeros((rows, cols, 3), dtype=torch.float64).pin_memory()
    pageable = np.ascontiguousarray(mm[1])
    ctx = pkg.Context(rows, cols)
    ctx.slam_init(np.zeros(6), xyz[0])
    pred, last, final = (p[0] for p in walk(2)[1])

    def refused(name, call, match):
        before = ctx.launch_count()
        with pytest.raises(pkg.NavError, match=match) as e:
            call()
        assert name in str(e.value), (name, str(e.value))
        assert ctx.launch_count() == before, name

    sub = "nav_frontend_submit_mm"
    refused(sub, lambda: ctx.frontend_submit_mm(pageable.ctypes.data, pred, last, final, global_out=out.data_ptr()),
            "pinned")
    refused("nav_slam_prefetch_mm", lambda: ctx.slam_prefetch(mm_ptr=pageable.ctypes.data), "pinned")
    for field, ptr in (("cloud", h_xyz[1].data_ptr()), ("distances", h_mm[1].data_ptr()),
                       ("cloud_out", out.data_ptr())):
        refused(sub, lambda: ctx.frontend_submit_mm(h_mm[1].data_ptr(), pred, last, final, **{field: ptr}),
                "must be NULL")
    ctx.set_tie_rule("reference")
    refused(sub, lambda: ctx.frontend_submit_mm(h_mm[1].data_ptr(), pred, last, final, global_out=out.data_ptr()),
            "tie rule")
    refused("nav_slam_run", lambda: ctx.slam_run([h_mm[1].data_ptr()], UNIT[None], np.zeros(6), mm_input=True),
            "tie rule")
    torch.cuda.synchronize()
    # the context still answers a supported call exactly: the blocking mm frame under the reference rule
    slam = oracle.slam(rows, cols, 0)
    slam.init(np.zeros(6), xyz[0])
    got = ctx.frontend_frame_mm(mm[1], pred, last, final)
    want = slam.frontend_frame(xyz[1], pred, last, final)
    for w, g in zip(want, got):
        assert np.array_equal(w, g)
    with pytest.raises(TypeError):
        ctx.frontend_frame_mm(xyz[1], pred, last, final)  # float input is not silently truncated
    slam.close()
    ctx.close()


@pytest.mark.gpu
def test_l9_csv_to_pinned_frames_to_submit_mm(pkg, synth, tmp_path):
    """the INTEGRATION.md path: reader -> int32 frames -> submit_mm, against the double reader -> submit"""
    import torch
    n = 4
    path = _write(tmp_path, synth.l9_csv(synth.l9_sequence(n)))
    mm, _ = pkg.l9_csv_read_mm(path, 16, 1800, n)
    xyz, _ = pkg.l9_csv_read(path, 16, 1800, n)
    h_mm, h_xyz = _pinned(mm), _pinned(xyz)
    res = []
    for kind in ("xyz", "mm"):
        ctx = pkg.Context(16, 1800)
        ctx.slam_init(np.zeros(6), xyz[0])
        idx = torch.zeros((n, 16, 1800), dtype=torch.int32).pin_memory()
        for f, (pred, last, final) in enumerate(walk(n, STEP)[1:], start=1):
            if kind == "xyz":
                ctx.frontend_submit(pred, last, final, cloud=h_xyz[f].data_ptr(), nn_idx_out=idx[f].data_ptr())
            else:
                ctx.frontend_submit_mm(h_mm[f].data_ptr(), pred, last, final, nn_idx_out=idx[f].data_ptr())
        ctx.frontend_wait()
        res.append(idx.numpy().copy())
        ctx.close()
    assert same(res[0], res[1]) and (res[1][1:] >= 0).any()
