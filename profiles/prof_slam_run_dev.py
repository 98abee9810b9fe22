#!/usr/bin/env python
"""The closed loop on device-resident frames (nav_slam_run_dev) at 64x2048 room data: microseconds per frame, timed
with CUDA events over at least 60 ms of work per line, next to
  - nav_slam_run (the host-driven loop) on pinned host frames, xyz and depth input,
  - nav_frontend_sequence_out_dev with fit_stats: the same per-frame work with the poses known, so the difference
    is the cost of the feedback,
  - the fit tail alone: %globaltimer stamps in the last CTA of each sequence, from a variant of the library built
    in a temporary directory with -DNAV_SEQ_TIMING (adding the partials, then the fit and the outputs).
Records the card's name and power limit.  usage: prof_slam_run_dev.py [out.txt]  (default profiles/r3_slam_run_dev.txt)
"""
import ctypes as C
import importlib
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
nav = importlib.import_module("nav-slam_b200")
synth = nav.synth

R, C_ = 64, 2048
NU = 40                 # distinct frames per sequence; longer runs repeat them (the set is far larger than L2)
F = 240                 # frames per call
MIN_MS = 60.0
STEP = np.array([48.0, 0.5, 0.0, 0.0, 0.0, 0.1])


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "power limit not readable"
    return f"{name}, power limit / max SM clock: {pl}"


def resident_frames(n_seq, n_frames):
    """[n_frames + 1][n_seq][R][C][3] on the device: frame 0 maps the context, 1.. are the loop (cycling NU frames)."""
    base = torch.from_numpy(np.stack([synth.room_sequence(R, C_, NU + 1, seq=s) for s in range(n_seq)], axis=1)).cuda()
    idx = torch.tensor([0] + [1 + (f % NU) for f in range(n_frames)], device="cuda")
    return base.index_select(0, idx).contiguous()


def timed(stream, fn, min_ms=MIN_MS, setup=None):
    """CUDA-event time of fn() on `stream`, summed over calls until min_ms: (ms per call, calls)."""
    total, calls = 0.0, 0
    while total < min_ms or calls < 3:
        if setup:
            setup()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        total += a.elapsed_time(b)
        calls += 1
    return total / calls, calls


def fit_tail_stamps(n_seq):
    """[frames][n_seq][4] %globaltimer stamps of the fit tail (variant library built with -DNAV_SEQ_TIMING)."""
    L = nav.load_library()
    L.nav_debug_set_loop_stamps.argtypes = [C.c_void_p]
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = nav.Context(R, C_, device=0, n_seq=n_seq)
    ctx.set_stream(stream.cuda_stream)
    fr = resident_frames(n_seq, F)
    deltas = np.tile(STEP, (F * n_seq, 1))
    z = np.zeros((n_seq, 6))
    out = torch.empty((F, n_seq, 6), dtype=torch.float64, device="cuda")
    stamps = torch.zeros((F, n_seq, 4), dtype=torch.int64, device="cuda")
    for rep in range(2):
        ctx.slam_init_dev(fr[0].data_ptr(), z)
        if rep == 1:
            assert L.nav_debug_set_loop_stamps(stamps.data_ptr()) == 0
        ctx.slam_run_dev(fr[1].data_ptr(), F, deltas, z, out.data_ptr())
        ctx.synchronize()
    assert L.nav_debug_set_loop_stamps(None) == 0
    ctx.close()
    return stamps.cpu().numpy()


def build_timing_variant(tmp):
    """libnavslam_b200.so with rowmap.cu compiled with -DNAV_SEQ_TIMING, the other objects from nav-slam_b200/_build."""
    b = nav.build
    b.build_library()
    obj = os.path.join(tmp, "rowmap.o")
    subprocess.check_call([b._nvcc(), *b.NVCC_FLAGS, "-DNAV_SEQ_TIMING", "-c", os.path.join(b.CSRC, "rowmap.cu"), "-o",
                           obj], stderr=subprocess.DEVNULL)
    objs = [obj if s == "rowmap.cu" else os.path.join(b.BUILD, s.replace(".cu", ".o")) for s in b.CU_SOURCES]
    lib = os.path.join(tmp, "libnavslam_b200.so")
    subprocess.check_call([b._nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib, *objs])
    return lib


def main_fit_tail():
    lines = []
    for n_seq in (1, 8):
        t = fit_tail_stamps(n_seq).astype(np.float64)[5:]   # skip the first frames
        add = (t[..., 1] - t[..., 0]).ravel() * 1e-3
        fit = (t[..., 2] - t[..., 1]).ravel() * 1e-3
        lines.append(f"  n_seq={n_seq}: adding the {R * C_ // 256} partials {np.median(add):6.2f} us (median; mean "
                     f"{add.mean():.2f}), fit (200 Adam iterations on one thread) + outputs + next record "
                     f"{np.median(fit):6.2f} us (median; mean {fit.mean():.2f}, min {fit.min():.2f}, max {fit.max():.2f}) "
                     f"over {fit.size} fits")
    print("\n".join(lines))


def main(out_path):
    lines = [f"prof_slam_run_dev.py: 64x2048 room data, CUDA events over >= {MIN_MS:.0f} ms per line", card(), ""]

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    for s in lines[:2]:
        print(s, flush=True)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)

    # nav_slam_run_dev, n_seq = 1, 2, 4, 8
    dev_us = {}
    for n_seq in (1, 2, 4, 8):
        ctx = nav.Context(R, C_, device=0, n_seq=n_seq)
        ctx.set_stream(stream.cuda_stream)
        fr = resident_frames(n_seq, F)
        deltas = np.tile(STEP, (F * n_seq, 1))
        z = np.zeros((n_seq, 6))
        poses = torch.empty((F, n_seq, 6), dtype=torch.float64, device="cuda")
        err = torch.empty((F, n_seq), dtype=torch.float64, device="cuda")
        st = torch.empty((F, n_seq, 5), dtype=torch.float64, device="cuda")
        run = lambda: ctx.slam_run_dev(fr[1].data_ptr(), F, deltas, z, poses.data_ptr(), err.data_ptr(), st.data_ptr())
        init = lambda: ctx.slam_init_dev(fr[0].data_ptr(), z)
        init()
        run()   # warm-up (scratch, tables)
        torch.cuda.synchronize()
        ms, calls = timed(stream, run, setup=init)
        us = ms * 1e3 / F
        dev_us[n_seq] = us
        p = poses.cpu().numpy()
        emit(f"nav_slam_run_dev n_seq={n_seq}: {us:7.2f} us per launch step ({F} frames x {n_seq} sequences per call, "
             f"{calls} calls) = {us / n_seq:6.2f} us per frame of one sequence = {n_seq * 1e6 / us:8.0f} frames/s; "
             f"last pose x = {p[-1, 0, 0]:.3f} mm, N = {int(st.cpu().numpy()[-1, 0, 0])}")
        if n_seq == 1:
            d_poses = p[:, 0]
        ctx.close()
        del fr

    # nav_slam_run on pinned host frames, xyz and depth
    clouds = synth.room_sequence(R, C_, NU + 1)
    frames = torch.from_numpy(clouds).pin_memory()
    depth = torch.from_numpy(np.stack([synth.l5_depth_frame(f, R, C_) for f in range(8)])).pin_memory()
    ctx = nav.Context(R, C_, device=0)
    ctx.set_stream(stream.cuda_stream)
    for use_depth in (False, True):
        src = depth if use_depth else frames
        ptrs = [src[1 + (f % (src.shape[0] - 1))].data_ptr() for f in range(F)]
        dl = np.tile(np.array([-19.0, 0.3, 0, 0, 0, 0]) if use_depth else STEP, (F, 1))
        init = lambda: ctx.slam_init(np.zeros(6), clouds[0], want_global=False)
        run = lambda: ctx.slam_run(ptrs, dl, np.zeros(6), depth_input=use_depth)
        init()
        run()
        ctx.synchronize()
        t0 = time.perf_counter()
        ms, calls = timed(stream, run, setup=init)
        wall = time.perf_counter() - t0
        us = ms * 1e3 / F
        emit(f"nav_slam_run {'depth' if use_depth else 'xyz  '} (pinned host frames): {us:7.2f} us per frame "
             f"= {1e6 / us:8.0f} frames/s ({F} frames, {calls} calls; wall {wall * 1e6 / (F * calls):.2f} us per frame "
             f"incl. the re-init between calls)")
    ctx.close()

    # the same work with known poses: nav_frontend_sequence_out_dev with fit_stats, poses from the device loop
    for n_seq in (1, 8):
        ctx = nav.Context(R, C_, device=0, n_seq=n_seq)
        ctx.set_stream(stream.cuda_stream)
        fr = resident_frames(n_seq, F)
        final = np.repeat(d_poses[:, None], n_seq, axis=1)
        last = np.concatenate([np.zeros((1, n_seq, 6)), final[:-1]])
        pred = last + STEP
        st = torch.empty((F, n_seq, 5), dtype=torch.float64, device="cuda")
        z = np.zeros((n_seq, 6))
        init = lambda: ctx.slam_init_dev(fr[0].data_ptr(), z)
        run = lambda: ctx.frontend_sequence_out_dev(fr[1].data_ptr(), F, pred.reshape(-1, 6), last.reshape(-1, 6),
                                                    final.reshape(-1, 6), fit_stats=st.data_ptr())
        init()
        run()
        torch.cuda.synchronize()
        ms, calls = timed(stream, run, setup=init)
        us = ms * 1e3 / F
        emit(f"nav_frontend_sequence_out_dev (known poses, fit_stats) n_seq={n_seq}: {us:7.2f} us per frame step = "
             f"{n_seq * 1e6 / us:8.0f} frames/s; device loop minus this: {dev_us[n_seq] - us:+6.2f} us per step")
        ctx.close()
        del fr

    # the fit tail alone, from the timing variant in a subprocess
    with tempfile.TemporaryDirectory() as tmp:
        lib = build_timing_variant(tmp)
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--fit-tail"], capture_output=True, text=True,
                           env={**os.environ, "NAVSLAM_LIB": lib})
        if r.returncode != 0:
            raise RuntimeError(r.stderr[-2000:])
        emit("fit tail of nav_slam_run_dev (last CTA of a sequence, %globaltimer, -DNAV_SEQ_TIMING build):")
        for s in r.stdout.rstrip().splitlines():
            emit(s)
    with open(out_path, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    if "--fit-tail" in sys.argv:
        main_fit_tail()
    else:
        main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_slam_run_dev.txt"))
