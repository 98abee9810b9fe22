#!/usr/bin/env python
"""Cost of replaying and closing the loop on depth and integer-mm recordings resident in HBM, against the same
recordings widened to xyz doubles, at 64x2048 on seeded room frames (synth.room_sequence, as bench.py; depth =
clip(|xyz|, 1, 60000) as bench.py forms it, integer mm = binding.to_mm of the rounded room).

Each kind is timed against the xyz replay of the cloud its frames stand for.
Replay (nav_frontend_sequence_dev / _dev_ex, one sequence, one k_frame_seq launch): K = 20 and K = 64 frames, without
and with all four per-frame rings.  Closed loop (nav_slam_run_dev / _dev_ex): 20 frames, 1 and 8 sequences.  The three
kinds alternate call by call; each call starts from a freshly initialised map; CUDA events time the call alone.  Every
variant gets at least 200 ms of device time per round, three rounds.  Printed: us per frame (all sequences of a
frame), the bytes of one frame of the recording, and the card's name, power limit and SM clock (sampled during the
run).  usage: prof_seq_inputs.py [min_ms_per_variant]"""
import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
nav = importlib.import_module("nav-slam_b200")
from prof_seq_outputs import gpu_info, start_clock_sampler, stop_clock_sampler  # noqa: E402

R, C_ = 64, 2048
MIN_MS = float(sys.argv[1]) if len(sys.argv) > 1 else 200.0
ROUNDS = 3
PRED_ERR = np.array([2.0, -1.0, 0.5, 0.0, 0.0, 0.05])
KINDS = ("depth", "xyz of depth", "mm", "xyz of mm")
RINGS = ("label_mask", "nn_idx", "nn_dist", "fit_stats")


def recordings(n_seq, k):
    """The recording as depth and as integer mm, and each widened to the xyz cloud it stands for (nav_convert_to_pointcloud
    of every depth image, float64 of the mm values): [k+1][n_seq][rows][cols](...) on the device.  A kind is compared
    with the xyz replay of its own cloud -- the depth cloud (x = range, the reference's field of view) is a different
    scene from the room's xyz, with other labels and searches."""
    xyz = np.stack([nav.synth.room_sequence(R, C_, k + 1, cfg=3, seq=s) for s in range(n_seq)], axis=1)
    depth = np.clip(np.linalg.norm(xyz, axis=-1), 1, 60000).astype(np.int32)
    mm = nav.to_mm(np.round(xyz) + 0.0)   # + 0.0: no -0.0, which to_mm refuses
    conv = nav.Context(R, C_, device=0)
    depth_xyz = np.stack([conv.convert_to_pointcloud(d) for d in depth.reshape(-1, R, C_)]).reshape(depth.shape + (3,))
    conv.close()
    dev = {"depth": depth, "xyz of depth": depth_xyz, "mm": mm, "xyz of mm": mm.astype(np.float64)}
    return {kd: torch.from_numpy(np.ascontiguousarray(dev[kd])).cuda() for kd in KINDS}


def kw(kind):
    return {"depth_input": kind == "depth", "mm_input": kind == "mm"}


def timed(stream, variants, reps):
    """reps calls of every variant, alternating; returns device ms per variant"""
    ev = {v: [] for v in variants}
    for _ in range(reps):
        for v, (prep, call) in variants.items():
            prep()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            call()
            e1.record(stream)
            ev[v].append((e0, e1))
    stream.synchronize()
    return {v: sum(a.elapsed_time(b) for a, b in ev[v]) for v in ev}


def rounds(label, stream, variants, frames_per_call):
    timed(stream, variants, 3)   # warm-up: module load, scratch growth
    ms1 = timed(stream, variants, 5)
    reps = max(5, int(np.ceil(MIN_MS / min(ms1[v] / 5 for v in ms1))))
    rows = []
    for rnd in range(ROUNDS):
        ms = timed(stream, variants, reps)
        rows.append({v: ms[v] / (reps * frames_per_call) * 1e3 for v in ms})
        print(f"  {label} round {rnd + 1}: {reps} calls per variant, "
              f"{min(ms.values()):.0f}-{max(ms.values()):.0f} ms of device time each", flush=True)
    return rows


def replay(k, with_rings, stream):
    d = recordings(1, k)
    ctx = nav.Context(R, C_, device=0)
    ctx.set_stream(stream.cuda_stream)
    rings = {"label_mask": torch.empty((k, R, C_ // 16), dtype=torch.int32, device="cuda"),
             "nn_idx": torch.empty((k, R, C_), dtype=torch.int32, device="cuda"),
             "nn_dist": torch.empty((k, R, C_), dtype=torch.float64, device="cuda"),
             "fit_stats": torch.empty((k, 5), dtype=torch.float64, device="cuda")}
    out = {f: rings[f].data_ptr() for f in RINGS} if with_rings else {}
    final = np.array([[50.0 * f, 0, 0, 0, 0, 0] for f in range(1, k + 1)])
    last = final - np.array([50.0, 0, 0, 0, 0, 0])
    pred = final + PRED_ERR
    z = np.zeros(6)
    variants = {}
    for kd in KINDS:
        variants[kd] = (lambda kd=kd: ctx.slam_init_dev(d[kd][0].data_ptr(), z, **kw(kd)),
                        lambda kd=kd: ctx.frontend_sequence_out_dev(d[kd][1].data_ptr(), k, pred, last, final, **out,
                                                                    **kw(kd)))
    rows = rounds(f"replay K={k} rings={'all' if with_rings else 'none'}", stream, variants, k)
    ctx.close()
    return rows


def closed_loop(n_seq, k, stream):
    d = recordings(n_seq, k)
    ctx = nav.Context(R, C_, device=0, n_seq=n_seq)
    ctx.set_stream(stream.cuda_stream)
    poses = torch.empty((k, n_seq, 6), dtype=torch.float64, device="cuda")
    err = torch.empty((k, n_seq), dtype=torch.float64, device="cuda")
    st = torch.empty((k, n_seq, 5), dtype=torch.float64, device="cuda")
    deltas = np.tile(np.array([50.0, 0, 0, 0, 0, 0]) + PRED_ERR, (k * n_seq, 1))
    z = np.zeros((n_seq, 6))
    variants = {}
    for kd in KINDS:
        variants[kd] = (lambda kd=kd: ctx.slam_init_dev(d[kd][0].data_ptr(), z, **kw(kd)),
                        lambda kd=kd: ctx.slam_run_dev(d[kd][1].data_ptr(), k, deltas, z, poses.data_ptr(),
                                                       err.data_ptr(), st.data_ptr(), **kw(kd)))
    rows = rounds(f"closed loop n_seq={n_seq} K={k}", stream, variants, k)
    ctx.close()
    return rows


def main():
    if nav.device_count() == 0:
        raise SystemExit("prof_seq_inputs.py: no CUDA device")
    stream = torch.cuda.Stream()
    print(f"GPU: {gpu_info()}  (name, power limit, max SM clock)", flush=True)
    sampler = start_clock_sampler()
    results = []
    try:
        for k in (20, 64):
            for with_rings in (False, True):
                results.append((f"replay, 1 sequence, K = {k}, rings: {'all four' if with_rings else 'none'}",
                                replay(k, with_rings, stream)))
        for n_seq in (1, 8):
            results.append((f"closed loop nav_slam_run_dev[_ex], {n_seq} sequence(s), K = 20", closed_loop(n_seq, 20, stream)))
    finally:
        clock = stop_clock_sampler(sampler)
    print(f"SM clock during the run: {clock}")
    print(f"bytes of one {R}x{C_} image: xyz {R * C_ * 24}, depth {R * C_ * 4}, mm {R * C_ * 12}")
    print("us per frame (all sequences of the frame), median of the rounds [min-max]; change against xyz")
    for label, rows in results:
        med = {kd: float(np.median([r[kd] for r in rows])) for kd in KINDS}
        cells = []
        for kd in KINDS:
            lo, hi = min(r[kd] for r in rows), max(r[kd] for r in rows)
            rel = f" ({(med[kd] / med['xyz of ' + kd] - 1) * 100:+.1f} % against xyz of {kd})" if kd in ("depth", "mm") else ""
            cells.append(f"{kd} {med[kd]:.2f} [{lo:.2f}-{hi:.2f}]{rel}")
        print(f"{label}:\n    " + "\n    ".join(cells))

if __name__ == "__main__":
    main()
