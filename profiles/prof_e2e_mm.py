#!/usr/bin/env python
"""Integer-mm input against xyz input, host buffers in and out, on one GPU.

Workloads: integer-mm 64x2048 room frames (synth.room_sequence(..., integer_mm=True)) and 16x1800 L9 frames
(synth.l9_sequence).  The int32 frames are np.rint of the synthetic clouds, the xyz frames their float64 widening,
so both arms compute the same outputs.
  e2e          nav_frontend_submit (xyz, 24 B/point in) against nav_frontend_submit_mm (int32, 12 B/point in), "masks"
               outputs (label masks + nn_idx + nn_dist), bench.py's e2e_leg method: wall clock around the submissions,
               drained with nav_frontend_wait, warmed up, at least MIN_MS per measurement.  The two arms alternate,
               ROUNDS rounds; the median round is printed.
  PCIe floor   the bare copies of one frame: H2D of the input (12 or 24 B/point) with the D2H of the masks outputs in
               flight on a second stream, one cudaMemcpyAsync per direction and frame; device time (CUDA events) of
               batches queued behind a sleep kernel.
  closed loop  nav_slam_run us/frame for xyz, mm and depth-matrix frames (prediction = last + true step + an error).
  widen        k_widen_mm device time per frame from a separate torch.profiler run.
The card's name, power limit and SM clock (sampled during the timed runs) are printed with the numbers.
usage: prof_e2e_mm.py [--out FILE] [--min-ms 60]"""
import argparse
import ctypes as C
import importlib
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
nav = importlib.import_module("nav-slam_b200")
NavFrameIO = nav.binding.NavFrameIO
NavPos = nav.binding.NavPos

ROUNDS = 5
N_RES = 16  # resident host frames, walked forwards and backwards
PRED_ERR = np.array([2.0, -1.0, 0.5, 0.0, 0.0, 0.05])


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


def pose_of(f):
    return np.array([50.0 * f, 0, 0, 0, 0, 0], dtype=np.float64)


def triangle(i, n):
    period = 2 * (n - 1)
    i %= period
    return i if i < n else period - i


# the CUDA runtime torch has loaded: the PCIe floor is timed on bare cudaMemcpyAsync calls
_CUDART = C.CDLL("libcudart.so.12")
_CUDART.cudaMemcpyAsync.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
H2D, D2H = 1, 2  # cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost


def memcpy_async(dst, src, nbytes, kind, stream):
    rc = _CUDART.cudaMemcpyAsync(dst, src, nbytes, kind, stream.cuda_stream)
    if rc != 0:
        raise RuntimeError(f"cudaMemcpyAsync failed: error {rc}")


def pos_c(p):
    return NavPos(*[float(v) for v in p])


class Shape:
    def __init__(self, name, rows, cols, clouds):
        self.name, self.rows, self.cols = name, rows, cols
        self.npx = rows * cols
        self.nch = (cols + 15) // 16
        mm = np.ascontiguousarray(np.rint(clouds).astype(np.int32))
        self.h_mm = torch.from_numpy(mm).pin_memory()
        self.h_xyz = torch.from_numpy(mm.astype(np.float64)).pin_memory()
        depth = np.clip(np.rint(np.linalg.norm(mm.astype(np.float64), axis=-1)), 1, 60000).astype(np.int32)
        self.h_depth = torch.from_numpy(depth).pin_memory()
        self.out_bytes = self.npx * 12 + rows * self.nch * 4  # nn_idx + nn_dist + label masks
        self.h_out = [torch.empty(self.out_bytes, dtype=torch.uint8).pin_memory() for _ in range(2)]
        self.ctx = nav.Context(rows, cols)
        self.L = self.ctx.L
        self.d_spin = torch.zeros((64, rows, cols, 3), dtype=torch.float64, device="cuda")
        self.d_spin_lab = torch.zeros((64, rows, cols), dtype=torch.int32, device="cuda")

    def spin_up(self, seconds=0.25):
        t_end = time.perf_counter() + seconds
        while time.perf_counter() < t_end:
            for _ in range(10):
                self.ctx.extract_feature_batch_dev(self.d_spin.data_ptr(), 64, self.d_spin_lab.data_ptr())
            torch.cuda.synchronize()

    def init_map(self):
        self.ctx.slam_init(pose_of(0), self.h_xyz[0].numpy(), want_global=False)

    def submit_step(self, kind):
        ios, pos = {}, {}
        L, h = self.L, self.ctx.h

        def step(i):
            cur, prev = triangle(i, N_RES), triangle(i - 1, N_RES)
            b = i & 1
            if b not in ios:
                p0 = self.h_out[b].data_ptr()
                io = NavFrameIO()
                io.nn_idx_out, io.nn_dist_out, io.mask_out = p0, p0 + self.npx * 4, p0 + self.npx * 12
                ios[b] = io
            if (prev, cur) not in pos:
                pos[(prev, cur)] = tuple(pos_c(p) for p in (pose_of(cur) + PRED_ERR, pose_of(prev), pose_of(cur)))
            pp, pl, pf = pos[(prev, cur)]
            if kind == "mm":
                rc = L.nav_frontend_submit_mm(h, self.h_mm[cur].data_ptr(), C.byref(ios[b]), C.byref(pp),
                                              C.byref(pl), C.byref(pf))
            else:
                ios[b].cloud = self.h_xyz[cur].data_ptr()
                rc = L.nav_frontend_submit(h, C.byref(ios[b]), C.byref(pp), C.byref(pl), C.byref(pf))
            if rc != 0:
                raise nav.NavError(L.nav_last_error().decode())
        return step

    def timed_wall(self, step, n_steps, warm=20):
        self.spin_up()
        self.init_map()
        for i in range(1, warm + 1):
            step(i)
        self.ctx.frontend_wait()
        t0 = time.perf_counter()
        for i in range(warm + 1, warm + 1 + n_steps):
            step(i)
        self.ctx.frontend_wait()
        return time.perf_counter() - t0

    def e2e_us(self, kind, min_ms):
        step = self.submit_step(kind)
        probe = self.timed_wall(step, 50) / 50
        n = int(max(50, np.ceil(min_ms * 1e-3 / probe)))
        return 1e6 * self.timed_wall(step, n) / n, n

    def pcie_floor_us(self, in_bytes, min_ms, slots=8, batch=256):
        """device time of `batch` frames of bare copies, one cudaMemcpyAsync per direction and frame: the H2D of
        in_bytes on one stream, the D2H of the masks outputs on another.  Both streams are held behind a sleep kernel
        while the host queues the batch, so the copies run back to back and the host's per-call cost stays out of the
        number."""
        h_in = torch.empty(in_bytes * slots, dtype=torch.uint8).pin_memory()
        d_in = torch.empty(in_bytes * slots, dtype=torch.uint8, device="cuda")
        h_out = torch.empty(self.out_bytes * slots, dtype=torch.uint8).pin_memory()
        d_out = torch.empty(self.out_bytes * slots, dtype=torch.uint8, device="cuda")
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        ob = self.out_bytes
        total_ms, frames = 0.0, 0
        while total_ms < min_ms or frames < 2 * batch:
            start = torch.cuda.Event(enable_timing=True)
            ends = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            with torch.cuda.stream(s1):
                torch.cuda._sleep(50_000_000)  # ~25 ms at 2 GHz: longer than queueing the batch takes
                start.record(s1)
            s2.wait_event(start)
            for i in range(batch):
                k = i % slots
                memcpy_async(d_in.data_ptr() + k * in_bytes, h_in.data_ptr() + k * in_bytes, in_bytes, H2D, s1)
                memcpy_async(h_out.data_ptr() + k * ob, d_out.data_ptr() + k * ob, ob, D2H, s2)
            ends[0].record(s1)
            ends[1].record(s2)
            torch.cuda.synchronize()
            total_ms += max(start.elapsed_time(e) for e in ends)
            frames += batch
        return 1e3 * total_ms / frames, in_bytes

    def slam_run_us(self, kind, min_ms):
        src = {"xyz": self.h_xyz, "mm": self.h_mm, "depth": self.h_depth}[kind]

        def run(n):
            seq = [triangle(i, N_RES) for i in range(n + 1)]
            ptrs = [src[f].data_ptr() for f in seq[1:]]
            deltas = np.stack([pose_of(seq[t + 1]) - pose_of(seq[t]) + np.array([-2.0, 0.5, 0, 0, 0, 0])
                               for t in range(n)])
            self.spin_up()
            self.init_map()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            self.ctx.slam_run(ptrs, deltas, pose_of(0), depth_input=kind == "depth", mm_input=kind == "mm")
            return (time.perf_counter() - t0) / n

        probe = run(100)
        n = int(max(200, np.ceil(min_ms * 1e-3 / probe)))
        return 1e6 * run(n), n

    def widen_us(self, n=200):
        from torch.profiler import ProfilerActivity, profile
        step = self.submit_step("mm")
        self.init_map()
        for i in range(1, 21):
            step(i)
        self.ctx.frontend_wait()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(21, 21 + n):
                step(i)
            self.ctx.frontend_wait()
        ev = [e for e in prof.key_averages() if "k_widen_mm" in e.key]
        if not ev:
            raise RuntimeError("k_widen_mm not found in the profile")
        total_us = sum(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) for e in ev)
        count = sum(e.count for e in ev)
        return total_us / count, count


def med(v):
    return float(np.median(v))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--min-ms", type=float, default=60.0)
    args = ap.parse_args()
    shapes = [Shape("room 64x2048 integer-mm", 64, 2048,
                    nav.synth.room_sequence(64, 2048, N_RES, integer_mm=True)),
              Shape("L9 16x1800", 16, 1800, nav.synth.l9_sequence(N_RES))]
    lines = [f"# profiles/prof_e2e_mm.py -- {gpu_info()} (name, power limit, max SM clock)",
             f"# e2e and nav_slam_run: wall clock, drained; PCIe floor: device time of queued copies; >= {args.min_ms:.0f} ms "
             f"per measurement, median of {ROUNDS} alternating rounds"]
    sampler = start_clock_sampler()
    res = {}
    for s in shapes:
        r = res[s.name] = {k: [] for k in ("e2e_xyz", "e2e_mm", "floor_xyz", "floor_mm", "run_xyz", "run_mm",
                                          "run_depth")}
        for _ in range(ROUNDS):
            for kind in ("xyz", "mm"):
                r["e2e_" + kind].append(s.e2e_us(kind, args.min_ms)[0])
                r["floor_" + kind].append(s.pcie_floor_us(s.npx * (24 if kind == "xyz" else 12), args.min_ms)[0])
            for kind in ("xyz", "mm", "depth"):
                r["run_" + kind].append(s.slam_run_us(kind, args.min_ms)[0])
    clock = stop_clock_sampler(sampler)
    lines.append(f"# SM clock during the timed runs: {clock}")
    for s in shapes:
        r = res[s.name]
        w_us, w_n = s.widen_us()
        mb_in = lambda b: s.npx * b / 1e6  # noqa: E731
        lines += [
            f"{s.name}: in {mb_in(24):.2f} MB (xyz) / {mb_in(12):.2f} MB (int32) per frame, out {s.out_bytes / 1e6:.2f} MB "
            f"(masks + nn_idx + nn_dist)",
            f"  e2e submit        xyz {med(r['e2e_xyz']):7.1f} us/frame   PCIe floor (24 B/pt H2D + D2H) "
            f"{med(r['floor_xyz']):6.1f} us",
            f"  e2e submit_mm     mm  {med(r['e2e_mm']):7.1f} us/frame   PCIe floor (12 B/pt H2D + D2H) "
            f"{med(r['floor_mm']):6.1f} us   speed-up {med(r['e2e_xyz']) / med(r['e2e_mm']):.2f}x",
            f"  rounds e2e xyz {[round(v, 1) for v in r['e2e_xyz']]}  mm {[round(v, 1) for v in r['e2e_mm']]}",
            f"  nav_slam_run      xyz {med(r['run_xyz']):7.1f}   mm {med(r['run_mm']):7.1f}   depth "
            f"{med(r['run_depth']):7.1f} us/frame",
            f"  k_widen_mm        {w_us:.2f} us/frame device time (torch.profiler, {w_n} launches; "
            f"{s.npx * 36 / 1e6:.2f} MB of HBM traffic per frame = {s.npx * 36 / (w_us * 1e-6) / 1e12:.2f} TB/s)",
        ]
    text = "\n".join(lines) + "\n"
    sys.stdout.write(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)
    for s in shapes:
        s.ctx.close()


if __name__ == "__main__":
    main()
