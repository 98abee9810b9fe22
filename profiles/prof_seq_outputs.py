#!/usr/bin/env python
"""Cost of keeping every frame's results of a device-resident sequence replay (nav_frontend_sequence_out_dev)
against nav_frontend_sequence_dev, at 64x2048 on seeded room frames (synth.room_sequence, as bench.py):
one sequence of K = 20 and K = 64 frames (one launch), and eight sequences side by side (the per-frame path).

Variants, alternating call by call: the plain replay; outputs {label_mask, nn_idx, nn_dist}; those + fit_stats;
fit_stats only.  Each call replays from a freshly initialised map; CUDA events time the replay call alone.  Every
variant gets at least 200 ms of device time per round, three rounds.  Printed: us per frame, frames/s, the bytes
the rings receive per frame, and the card's name, power limit and SM clock (sampled during the run).
usage: prof_seq_outputs.py [min_ms_per_variant]"""
import importlib
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
nav = importlib.import_module("nav-slam_b200")

R, C_ = 64, 2048
MIN_MS = float(sys.argv[1]) if len(sys.argv) > 1 else 200.0
ROUNDS = 3
PRED_ERR = np.array([2.0, -1.0, 0.5, 0.0, 0.0, 0.05])
VARIANTS = [("sequence_dev", ()), ("outputs", ("label_mask", "nn_idx", "nn_dist")),
            ("outputs+stats", ("label_mask", "nn_idx", "nn_dist", "fit_stats")), ("stats only", ("fit_stats",))]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


def start_clock_sampler():
    try:
        return subprocess.Popen(["nvidia-smi", "--id=0", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits",
                                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except OSError:
        return None


def stop_clock_sampler(p):
    if p is None:
        return "not sampled"
    p.terminate()
    out, _ = p.communicate(timeout=10)
    mhz = [float(v) for v in out.split() if v.replace(".", "").isdigit()]
    hi = [v for v in mhz if mhz and v >= 0.5 * max(mhz)]
    return f"{np.median(hi):.0f} MHz (median of {len(hi)} loaded samples of {len(mhz)})" if hi else "not sampled"


def workload(n_seq, k):
    frames = np.stack([nav.synth.room_sequence(R, C_, k + 1, cfg=3, seq=s) for s in range(n_seq)], axis=1)
    final = np.array([[[50.0 * f, 2.0 * s, 0, 0, 0, 0] for s in range(n_seq)] for f in range(1, k + 1)])
    last = np.array([[[50.0 * (f - 1), 2.0 * s, 0, 0, 0, 0] for s in range(n_seq)] for f in range(1, k + 1)])
    return torch.from_numpy(np.ascontiguousarray(frames)).cuda(), final + PRED_ERR, last, final


def ring_bytes(n_seq):
    """Bytes per frame each output field receives (algorithmic: what the caller keeps)."""
    return {"label_mask": n_seq * R * (C_ // 16) * 4, "nn_idx": n_seq * R * C_ * 4, "nn_dist": n_seq * R * C_ * 8,
            "fit_stats": n_seq * 5 * 8}


def measure(n_seq, k, stream):
    d_frames, pred, last, final = workload(n_seq, k)
    ctx = nav.Context(R, C_, device=0, n_seq=n_seq)
    ctx.set_stream(stream.cuda_stream)
    rings = {"label_mask": torch.empty((k, n_seq, R, C_ // 16), dtype=torch.int32, device="cuda"),
             "nn_idx": torch.empty((k, n_seq, R, C_), dtype=torch.int32, device="cuda"),
             "nn_dist": torch.empty((k, n_seq, R, C_), dtype=torch.float64, device="cuda"),
             "fit_stats": torch.empty((k, n_seq, 5), dtype=torch.float64, device="cuda")}
    args = (d_frames[1].data_ptr(), k, pred.reshape(-1, 6), last.reshape(-1, 6), final.reshape(-1, 6))
    z = np.zeros((n_seq, 6))

    def batch(reps):
        """reps calls of every variant, alternating; returns device ms per variant"""
        ev = {v: [] for v, _ in VARIANTS}
        for _ in range(reps):
            for v, fields in VARIANTS:
                ctx.slam_init_dev(d_frames[0].data_ptr(), z)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                ctx.frontend_sequence_out_dev(*args, **{f: rings[f].data_ptr() for f in fields})
                e1.record(stream)
                ev[v].append((e0, e1))
        stream.synchronize()
        return {v: sum(a.elapsed_time(b) for a, b in ev[v]) for v in ev}

    batch(3)                                   # warm-up: module load, scratch and pose-ring growth
    ms1 = batch(5)
    reps = max(5, int(np.ceil(MIN_MS / min(ms1[v] / 5 for v in ms1))))
    rows = []
    for rnd in range(ROUNDS):
        ms = batch(reps)
        rows.append({v: ms[v] / (reps * k) * 1e3 for v in ms})   # us per frame (all sequences of the frame)
        print(f"  n_seq={n_seq} K={k} round {rnd + 1}: {reps} calls per variant, "
              f"{min(ms.values()):.0f}-{max(ms.values()):.0f} ms of device time each", flush=True)
    ctx.close()
    return rows


def main():
    if nav.device_count() == 0:
        raise SystemExit("prof_seq_outputs.py: no CUDA device")
    stream = torch.cuda.Stream()
    print(f"GPU: {gpu_info()}  (name, power limit, max SM clock)", flush=True)
    sampler = start_clock_sampler()
    results = {}
    try:
        for n_seq, k in ((1, 20), (1, 64), (8, 20)):
            results[(n_seq, k)] = measure(n_seq, k, stream)
    finally:
        clock = stop_clock_sampler(sampler)
    print(f"SM clock during the run: {clock}")
    for (n_seq, k), rows in results.items():
        rb = ring_bytes(n_seq)
        path = "one launch" if n_seq == 1 else "per-frame path"
        print(f"\n64x2048, n_seq={n_seq}, K={k} ({path}); us per frame of {n_seq} image(s), rounds 1-3 | median | "
              f"frames/s (images) | vs sequence_dev | ring bytes per frame")
        base = np.median([r["sequence_dev"] for r in rows])
        for v, fields in VARIANTS:
            us = [r[v] for r in rows]
            med = float(np.median(us))
            nb = sum(rb[f] for f in fields)
            print(f"  {v:14s} {' '.join(f'{u:7.2f}' for u in us)} | {med:7.2f} | {n_seq * 1e6 / med:9.0f} | "
                  f"{(med / base - 1) * 100:+6.1f} % | {nb / 1e6:6.3f} MB" + (f" ({nb / med / 1e3:.0f} GB/s)" if nb else ""))


if __name__ == "__main__":
    main()
