#!/usr/bin/env python
"""bench.py -- NAV-SLAM front end on B200: frames/s (feature extract + NN match).

Workload (config.workload): BASELINE.json configs[2], the 64x2048 OS1-64-shaped range-image
sequence.  One step = one frame of the sequence through the front end in the reference's own
order (SURVEY 8d "one frame of work"): curvature/edge labels (a3), query transform (a7), exact
per-row nearest neighbour against the previous frame's labelled points (a6), then mapping with the
final pose: transform (a7), row compaction (a4) and per-row map build (a5).  Frames are processed
sequentially (frame t is matched against frame t-1), exactly like slam_localization +
slam_mapping; the Adam pose fit and the EKF stay on the host in the reference and are not part of
the metric (the whole step with pose feedback is reported beside it as `e2e_closed_loop`).

  value : frames/s with the sequence resident in HBM (nav_frontend_sequence_dev: one launch per frame,
          consecutive launches overlapped by programmatic dependent launch).  Exactly K = --steps steps
          are timed, after W = --warmup untimed ones, between one pair of CUDA events (three untimed
          passes over the same frames come first, so that their first device touch is not timed);
          `ms_per_step` is that time / K.  --dump-outputs DIR writes what the last timed step computed
          (labels, NN indices and distances, mapped cloud, map masks) as DIR/<name>.npy.
  e2e   : frames/s through the host-buffer C ABI call (nav_frontend_submit): every step copies the frame
          from pinned host memory to the device and copies the step's results -- labels, NN indices, NN
          distances -- back; uploads, kernels and downloads of consecutive frames overlap.
  roofline : the kernel with the largest share of the step, timed live with CUDA events
  cpu_baseline : the reference's own C functions (oracle/_ref, built from /root/reference) on one
          host core for a bounded sample of the same frames

`--impl reference` runs that CPU path alone on all host cores (one process per core, the
reference has no threads).  Multi-GPU (--gpus N under torchrun): independent sequences per rank
(config 5a), no data-path collective, weak scaling; the large-map queries sharded against a
replicated tree (config 5b) are reported under `nn`.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

ROWS, COLS = 64, 2048
NPX = ROWS * COLS
FRAME_BYTES = NPX * 24
L2_BYTES = 126 * 1024 * 1024
METRIC = "frames/sec (feature extract + NN match)"
# both arms print this string (the driver compares the configs of the two lines)
WORKLOAD = "cfg3: 64x2048 OS1-64-shaped sequence, feature extraction + scan matching, one independent sequence per GPU"


def load_pkg():
    return importlib.import_module("nav-slam_b200")


_REAL_STDOUT = None


def print_line(line):
    txt = json.dumps(line) + "\n"
    if _REAL_STDOUT is None:
        sys.stdout.write(txt)
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, txt.encode())


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops", 1590.0)), "measured"
    return 6650.0, 1590.0, "fallback"


# ------------------------------------------------------------------ clocks ----------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # median over the samples taken under load (the sampler also sees the idle gaps between legs)
        hi = [v for v in sm if mx and v >= 0.5 * max(mx)]
        return {"sm_mhz": float(np.median(hi or sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------ workload --------------------
def make_frames(pkg, n_frames: int, seq: int):
    return pkg.synth.room_sequence(ROWS, COLS, n_frames, cfg=3, seq=seq)


def pose_of(frame: int):
    return np.array([50.0 * frame, 0, 0, 0, 0, 0], dtype=np.float64)


PRED_ERR = np.array([2.0, -1.0, 0.5, 0.0, 0.0, 0.05])


def poses_between(prev: int, cur: int):
    """Step from resident frame `prev` to frame `cur`: prediction = odometry with a small error, final =
    ground truth (the sensor moves 50 mm per frame index along +x)."""
    final = pose_of(cur)
    return final + PRED_ERR, pose_of(prev), final


def poses_for(frame: int):
    return poses_between(frame - 1, frame)


def triangle(i: int, n: int) -> int:
    """Frame index of step i when the resident sequence is walked forwards and backwards for ever
    (0, 1, ..., n-1, n-2, ..., 0, 1, ...): every step moves to a neighbouring frame, so every step is an
    ordinary 50 mm step however long the timed region is."""
    period = 2 * (n - 1)
    i %= period
    return i if i < n else period - i


# ------------------------------------------------------------------ CPU reference arm -----------
def _ref_frames_worker(args):
    """Front end of `count` frames with the reference's own functions on one core."""
    seq, start, count = args
    from oracle_lib import Oracle, RefLib, ref_available
    pkg = load_pkg()
    use_ref = ref_available(f"{ROWS}x{COLS}")
    o = Oracle()
    frames = pkg.synth.room_sequence(ROWS, COLS, count + 1, cfg=3, seq=seq, start=start)
    if use_ref:
        ref = RefLib(ROWS, COLS)
        t_total = 0.0
        ph = {"a3_extract_feature": 0.0, "a7_transform": 0.0, "a6_nn_search": 0.0, "a4_a5_flatten_build": 0.0}
        feat_prev = ref.extract_feature(frames[0])
        g_prev = o.transform(frames[0], poses_for(start)[2])
        trees, _, _ = ref.build_rows(g_prev, feat_prev)
        for i in range(1, count + 1):
            pred, last, final = poses_for(start + i)
            t_feat = ref.time_extract_feature(frames[i], reps=1)                 # a3
            feat = ref.extract_feature(frames[i])
            t1 = time.perf_counter()
            q = o.shift(o.transform(frames[i], pred), pred[:3] - last[:3])         # a7 (restated; <1 ms)
            g = o.transform(frames[i], final)
            t2 = time.perf_counter()
            _, _, _, t_nn = ref.nn_rows(trees, q, feat)                             # a6
            ref.free_rows(trees)
            trees, _, t_build = ref.build_rows(g, feat)                             # a4 + a5
            t_total += t_feat + (t2 - t1) + t_nn + t_build
            ph["a3_extract_feature"] += t_feat
            ph["a7_transform"] += t2 - t1
            ph["a6_nn_search"] += t_nn
            ph["a4_a5_flatten_build"] += t_build
        ref.free_rows(trees)
        return t_total, count, "reference", {k: 1e3 * v / count for k, v in ph.items()}
    slam = o.slam(ROWS, COLS, 0)
    slam.init(poses_for(start)[2], frames[0])
    t0 = time.perf_counter()
    for i in range(1, count + 1):
        pred, last, final = poses_for(start + i)
        slam.frontend_frame(frames[i], pred, last, final)
    dt = time.perf_counter() - t0
    slam.close()
    return dt, count, "port", None


def _ref_whole_step_worker(n_frames):
    """The reference's slam_localization + slam_mapping (src/slam.c:178-431) with pose feedback, one core."""
    from oracle_lib import Pos, RefLib, quiet_stdout, ref_available
    if not ref_available(f"{ROWS}x{COLS}"):
        return None
    pkg = load_pkg()
    frames = pkg.synth.room_sequence(ROWS, COLS, n_frames + 1, cfg=3, seq=0)
    ref = RefLib(ROWS, COLS)
    attr = ref.new_attr()
    pc = [ref.pack_cloud(frames[f], ts=f) for f in range(n_frames + 1)]
    ref.lib.init_slam(attr.ctypes.data, Pos.of(np.zeros(6)), pc[0].ctypes.data)
    last = np.zeros(6)
    ts = []
    with quiet_stdout():
        for f in range(1, n_frames + 1):
            pred = last + np.array([48.0, 0.5, 0.0, 0.0, 0.0, 0.0])
            t0 = time.perf_counter()
            p = ref.lib.slam_localization(attr.ctypes.data, pc[f].ctypes.data, Pos.of(pred), Pos.of(last)).arr()
            ref.lib.slam_mapping(attr.ctypes.data, Pos.of(p), pc[f].ctypes.data)
            ts.append(time.perf_counter() - t0)
            last = p
    return float(np.median(ts))


def _preload_reference():
    """dlopen oracle/_ref in THIS process (the forked workers inherit the mapping), so that the process the
    driver watches shows which reference library the CPU arm runs."""
    try:
        from oracle_lib import RefLib, ref_available
        if ref_available(f"{ROWS}x{COLS}"):
            return RefLib(ROWS, COLS)
    except Exception:  # noqa: BLE001
        pass
    return None


def cpu_baseline_single_core(n_frames: int, whole_step_frames: int):
    _preload_reference()
    try:
        os.sched_setaffinity(0, {sorted(os.sched_getaffinity(0))[0]})
        pinned = True
    except (AttributeError, OSError):
        pinned = False
    import multiprocessing as mp
    with mp.get_context("fork").Pool(1) as pool:
        dt, cnt, kind, phases = pool.map(_ref_frames_worker, [(0, 0, n_frames)])[0]
        whole = pool.map(_ref_whole_step_worker, [whole_step_frames])[0] if whole_step_frames > 0 else None
    if pinned:
        os.sched_setaffinity(0, set(range(os.cpu_count() or 1)))
    return {"value": cnt / dt, "unit": "frames/s", "cores": 1, "kind": kind,
            "sample": f"{cnt} frames of the 64x2048 sequence; extract_feature + per-row flattenPoints/"
                      f"buildKDTree + nearestNeighborSearch per labelled point, one core",
            "ms_per_frame": 1e3 * dt / cnt, "phase_ms_per_frame": phases,
            "whole_step_ms_per_frame": None if whole is None else 1e3 * whole,
            "whole_step_note": "slam_localization + slam_mapping of the reference with pose feedback (O(n^2) dedupe and "
                               f"the 200 x N Adam loop included), median of {whole_step_frames} frames, one core"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    ref = _preload_reference()
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    per_worker = 2
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        def step(i):
            jobs = [(w, 10 * i, per_worker) for w in range(cores)]
            res = pool.map(_ref_frames_worker, jobs)
            # workers also generate their inputs; charge only the time spent inside the front end
            return max(r[0] for r in res), res[0][2]
        for i in range(args.warmup):
            step(i)
        tot = 0.0
        kind = "reference"
        for i in range(args.steps):
            busy, kind = step(args.warmup + i)
            tot += busy
    frames = args.steps * cores * per_worker
    v = frames / tot
    line = {
        "impl": "reference", "metric": METRIC, "value": v,
        "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "step": f"{cores} processes x {per_worker} frames each (bounded sample per step)"},
        "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "kind": kind,
                         "sample": f"{frames} frames, {cores} single-threaded processes",
                         "library": None if ref is None else os.path.relpath(ref.lib._name, ROOT)},
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print_line(line)


# ------------------------------------------------------------------ shim leg (child process) ----
def run_shim_leg(args):
    """e2e through the reference's OWN entry points (headers/slam.h:22-28) served by the per-shape shim:
    init_slam, then slam_localization + slam_mapping per frame with pose feedback, exactly the calls
    src/main.c:300-318 makes.  Runs in a child process because the shim reads NAVSLAM_ADAM / NAVSLAM_TRUST_FRAME
    once and prints the reference's per-iteration lines on stdout."""
    pkg = load_pkg()
    sb = importlib.import_module("nav-slam_b200.shim_binding")
    n = args.shim_frames
    frames = pkg.synth.room_sequence(ROWS, COLS, n + 1, cfg=3, seq=0)
    shim = sb.ShimSlam(ROWS, COLS)
    # ONE PointCloud buffer refilled for every frame, as the reference's handlers do (src/main.c:250,308)
    pc = shim.pack_cloud(frames[0], ts=0)

    def load(f):
        pc[:4] = np.frombuffer(np.int32(f).tobytes(), dtype=np.uint8)
        pc[8:] = frames[f].reshape(-1).view(np.uint8)
        return pc
    devnull = os.open(os.devnull, os.O_WRONLY)
    saved = os.dup(1)
    sys.stdout.flush()
    os.dup2(devnull, 1)
    try:
        shim.init_slam(np.zeros(6), load(0))
        last = np.zeros(6)
        ts = []
        for f in range(1, n + 1):
            pred = last + np.array([48.0, 0.5, 0.0, 0.0, 0.0, 0.0])
            load(f)
            t0 = time.perf_counter()
            p = shim.slam_localization(pc, pred, last)
            shim.slam_mapping(p, pc)
            ts.append(time.perf_counter() - t0)
            last = p
    finally:
        os.dup2(saved, 1)
        os.close(devnull)
    skip = min(3, n // 3)
    t = float(np.median(ts[skip:]))
    out = {"ms_per_frame": 1e3 * t, "frames_per_s": 1.0 / t, "frames": n, "pose_x": float(last[0]),
           "pose_x_truth": 50.0 * n, "rms_mm": shim.error,
           "NAVSLAM_ADAM": os.environ.get("NAVSLAM_ADAM", ""), "NAVSLAM_TRUST_FRAME": os.environ.get("NAVSLAM_TRUST_FRAME", ""),
           "NAVSLAM_PIN": os.environ.get("NAVSLAM_PIN", "")}
    with open(args.shim_out, "w") as f:
        json.dump(out, f)
    shim.release()


def shim_legs():
    """Both modes of the shim, each in its own process; {} if a leg fails."""
    out = {}
    for name, env, n in (("default", {}, 12),
                         ("stats", {"NAVSLAM_ADAM": "stats"}, 60),
                         ("stats_trust_frame", {"NAVSLAM_ADAM": "stats", "NAVSLAM_TRUST_FRAME": "1"}, 60),
                         ("stats_trust_frame_pinned", {"NAVSLAM_ADAM": "stats", "NAVSLAM_TRUST_FRAME": "1",
                                                       "NAVSLAM_PIN": "1"}, 60)):
        with tempfile.NamedTemporaryFile(suffix=".json", delete=False) as tf:
            path = tf.name
        e = dict(os.environ)
        for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "NAVSLAM_ADAM", "NAVSLAM_TRUST_FRAME", "NAVSLAM_PIN"):
            e.pop(k, None)
        e.update(env)
        try:
            subprocess.run([sys.executable, os.path.abspath(__file__), "--shim-leg", "--shim-out", path,
                            "--shim-frames", str(n)], env=e, check=True, timeout=300,
                           stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
            with open(path) as f:
                out[name] = json.load(f)
        except Exception as ex:  # noqa: BLE001
            out[name] = {"error": str(ex)[:300]}
        finally:
            try:
                os.unlink(path)
            except OSError:
                pass
    return out


def bind_near_gpu(torch, local):
    """Pin this rank to the CPU cores next to its GPU (NVML's CPU affinity of the device) before any
    pinned memory is allocated: first touch then places the staging buffers on the GPU's NUMA node, and
    eight ranks do not push their PCIe traffic through one socket.  Best effort; returns the core count."""
    try:
        import pynvml
        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(local)
        bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        words = pynvml.nvmlDeviceGetCpuAffinity(h, ((os.cpu_count() or 64) + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:  # noqa: BLE001 -- no NVML, no affinity API: run unbound
        pass
    return None


# ------------------------------------------------------------------ GPU arm ---------------------
class Raw:
    """n elements of a device buffer the library owns, for torch.as_tensor(..., device="cuda")."""
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


def dump_outputs(out_dir, res, torch):
    """What the timed path hands its caller for the last timed frame (nav_frame_results_dev), copied to the
    host: int32 labels as float32, indices and bit masks as float64 (exact), distances and the mapped cloud
    as float64.  5.8 MB in all."""
    n_chunks = (COLS + 15) // 16
    arrays = {"labels": (res.labels, (ROWS, COLS), "<i4", np.float32),
              "nn_idx": (res.nn_idx, (ROWS, COLS), "<i4", np.float64),
              "nn_dist": (res.nn_dist, (ROWS, COLS), "<f8", np.float64),
              "global_cloud": (res.global_, (ROWS, COLS, 3), "<f8", np.float64),
              "map_mask": (res.map_mask, (ROWS, n_chunks), "<i4", np.float64)}
    torch.cuda.synchronize()
    os.makedirs(out_dir, exist_ok=True)
    for name, (ptr, shape, typestr, np_dtype) in arrays.items():
        n = int(np.prod(shape))
        host = torch.as_tensor(Raw(ptr, n, typestr), device="cuda").cpu().numpy().reshape(shape)
        if name == "map_mask":
            host = host.view(np.uint32)        # 32-bit masks: read as unsigned
        np.save(os.path.join(out_dir, name + ".npy"), host.astype(np_dtype))


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cpu = None
    if rank == 0 and not args.skip_cpu:   # forks: do it before CUDA is initialised
        cpu = cpu_baseline_single_core(args.cpu_frames if world == 1 else min(args.cpu_frames, 20),
                                       args.cpu_whole_frames if world == 1 else 0)
    if world > 1:
        # NCCL prints its version banner on stdout at NCCL_DEBUG=VERSION; stdout carries the JSON line
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    bound_cores = bind_near_gpu(torch, local) if world > 1 else None
    pkg = load_pkg()
    if pkg.device_count() == 0:
        raise RuntimeError("bench.py: no CUDA device; the product has no CPU fallback")
    K, W = args.steps, args.warmup
    # the resident sequence is sized independently of --steps: always several times the L2
    n_res = max(args.frames, K + W + 2)
    frames = make_frames(pkg, n_res, seq=rank)  # [F,64,2048,3] fp64, 3.1 MB each
    L = pkg.load_library()
    binding = importlib.import_module("nav-slam_b200.binding")
    NavPos, NavFrameIO = binding.NavPos, binding.NavFrameIO
    ctx = pkg.Context(ROWS, COLS, device=local, n_seq=1)
    stream = torch.cuda.Stream()           # a real (non-default) stream: events and kernels share it
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)

    d_frames = torch.from_numpy(frames).cuda()
    h_frames = torch.from_numpy(frames).pin_memory()     # pinned host copies for the e2e legs
    d_base, h_base = d_frames.data_ptr(), h_frames.data_ptr()
    import ctypes as C

    def check(rc):
        if rc:
            raise RuntimeError(L.nav_last_error().decode())

    def pos_c(p):
        return NavPos(*[float(v) for v in p])

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(vals):
        if world == 1:
            return [float(v) for v in vals]
        t = torch.tensor(list(vals), device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    # a buffer of its own for keeping the clocks up: nothing the timed regions read goes through L2 here
    d_spin_in = torch.randn((24, ROWS, COLS, 3), dtype=torch.float64, device="cuda")
    d_spin_out = torch.empty((24, ROWS, COLS), dtype=torch.int32, device="cuda")

    def spin_up(seconds=0.25):
        """Keep the GPU busy so that the SM clocks are at their loaded level when a timed region starts
        (host-side input generation leaves the device idle for seconds)."""
        t_end = time.perf_counter() + seconds
        while time.perf_counter() < t_end:
            for _ in range(20):
                ctx.extract_feature_batch_dev(d_spin_in.data_ptr(), d_spin_in.shape[0], d_spin_out.data_ptr())
            torch.cuda.synchronize()

    def pose_block(first, count):
        arrs = [(NavPos * count)() for _ in range(3)]
        for i in range(count):
            for a, p in zip(arrs, poses_for(first + i)):
                a[i] = pos_c(p)
        return arrs

    # ---------------- value: device resident, the K timed steps on frames F0 + W .. F0 + W + K - 1
    F0 = 1
    p_init, wp, kp = pos_c(pose_of(F0 - 1)), pose_block(F0, W), pose_block(F0 + W, K)

    def run_window():
        """Re-initialise the map on frame F0 - 1, W untimed steps, then the K steps between two events.
        Returns their device ms and the launches of the whole window (re-init and warm-up included)."""
        barrier()
        l0 = ctx.launch_count()
        check(L.nav_slam_init_dev(ctx.h, d_base + (F0 - 1) * FRAME_BYTES, C.byref(p_init)))
        check(L.nav_frontend_sequence_dev(ctx.h, d_base + F0 * FRAME_BYTES, W, *wp))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        check(L.nav_frontend_sequence_dev(ctx.h, d_base + (F0 + W) * FRAME_BYTES, K, *kp))
        e1.record(stream)
        barrier()
        return e0.elapsed_time(e1), ctx.launch_count() - l0

    clocks = ClockSampler(local)
    clocks.start()
    spin_up()
    for _ in range(3):     # untimed passes over the same frames: their first device touch is not timed
        run_window()
    spin_up()
    dev_ms, window_launches = run_window()       # --steps is the number of timed steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx.frame_results_dev(), torch)
    if world > 1:
        per_rank = [None] * world
        dist.all_gather_object(per_rank, dev_ms / K)
    else:
        per_rank = [dev_ms / K]
    dev_ms = reduce_max([dev_ms])[0]

    # ---------------- per-kernel durations (CUDA events on the launching stream, one pair per launch)
    ctx.profile_enable(True)
    for name in ("labels", "match", "map"):
        ctx.profile_read(name, reset=True)
    spin_up()
    check(L.nav_slam_init_dev(ctx.h, d_base, C.byref(pos_c(pose_of(0)))))
    n_prof = min(n_res - 1, max(K, 64))
    for f in range(1, n_prof + 1):
        pp, pl, pf = (pos_c(p) for p in poses_for(f))
        check(L.nav_frontend_frame_dev(ctx.h, d_base + f * FRAME_BYTES, C.byref(pp), C.byref(pl), C.byref(pf)))
    prof = {name: ctx.profile_read(name, reset=True) for name in ("match", "map")}
    prof = {("frame_fused" if k == "match" else k): v for k, v in prof.items() if v[1]}
    ctx.profile_enable(False)

    # ---------------- e2e legs: host buffers in, host buffers out, through the C ABI
    n_chunks = (COLS + 15) // 16
    h_out = [torch.empty(NPX * 40 + ROWS * n_chunks * 4, dtype=torch.uint8).pin_memory() for _ in range(2)]
    # per-frame depth matrices for the L5-type input (utils/pointcloud.c:8): ranges of the same room
    h_depth = torch.from_numpy(np.ascontiguousarray(
        np.clip(np.linalg.norm(frames[: min(n_res, 128)], axis=-1), 1, 60000).astype(np.int32))).pin_memory()
    n_depth = int(h_depth.shape[0])

    def out_ptrs(b):
        p0 = h_out[b].data_ptr()
        return {"feature": p0, "idx": p0 + NPX * 4, "dist": p0 + NPX * 8, "global": p0 + NPX * 16,
                "mask": p0 + NPX * 40}

    def make_submit(kind):
        """Build the per-step callable of one e2e variant.  Steps walk the resident frames forwards and
        backwards (triangle), so the region can be as long as it needs to be."""
        ios, pos = {}, {}

        def step(i):
            cur, prev = triangle(i, n_res), triangle(i - 1, n_res)
            key = (cur, i & 1)
            if key not in ios:
                o = out_ptrs(i & 1)
                io = NavFrameIO()
                if kind in ("depth_masks", "depth_masks_idx"):
                    io.distances = h_depth.data_ptr() + (cur % n_depth) * NPX * 4
                else:
                    io.cloud = h_base + cur * FRAME_BYTES
                if kind in ("masks", "depth_masks", "depth_masks_idx"):
                    io.mask_out = o["mask"]
                else:
                    io.feature_out = o["feature"]
                io.nn_idx_out = o["idx"]
                if kind != "depth_masks_idx":
                    io.nn_dist_out = o["dist"]
                if kind == "all_outputs":
                    io.global_out = o["global"]
                ios[key] = io
            if (prev, cur) not in pos:
                pos[(prev, cur)] = tuple(pos_c(p) for p in poses_between(prev, cur))
            pp, pl, pf = pos[(prev, cur)]
            check(L.nav_frontend_submit(ctx.h, C.byref(ios[key]), C.byref(pp), C.byref(pl), C.byref(pf)))
        return step

    def blocking_step(i):
        cur, prev = triangle(i, n_res), triangle(i - 1, n_res)
        pp, pl, pf = (pos_c(p) for p in poses_between(prev, cur))
        o = out_ptrs(0)
        check(L.nav_frontend_frame(ctx.h, h_base + cur * FRAME_BYTES, C.byref(pp), C.byref(pl), C.byref(pf),
                                   o["feature"], o["idx"], o["dist"], o["global"]))

    def timed_wall(step_fn, n_steps, drain):
        """Wall clock around n_steps calls (several streams are involved), barrier + synchronize both sides."""
        spin_up()
        check(L.nav_slam_init_dev(ctx.h, d_base, C.byref(pos_c(pose_of(0)))))
        for i in range(1, W + 1):
            step_fn(i)
        if drain:
            drain()
        barrier()
        t0 = time.perf_counter()
        for i in range(W + 1, W + 1 + n_steps):
            step_fn(i)
        if drain:
            drain()
        barrier()
        wall = time.perf_counter() - t0
        return reduce_max([wall])[0]

    def e2e_leg(kind):
        fn = make_submit(kind)
        probe = timed_wall(fn, max(K, 20), ctx.frontend_wait) / max(K, 20)
        n_steps = int(min(20000, max(K, np.ceil(args.min_timed_ms * 1e-3 / probe))))
        wall = timed_wall(fn, n_steps, ctx.frontend_wait)
        return {"value": world * n_steps / wall, "unit": "frames/s", "steps_timed": n_steps,
                "wall_ms_per_step": 1e3 * wall / n_steps}

    e2e_masks = e2e_leg("masks")
    e2e_labels = e2e_leg("labels")
    e2e_all = e2e_leg("all_outputs")
    e2e_depth = e2e_leg("depth_masks")
    e2e_depth_idx = e2e_leg("depth_masks_idx")
    n_block = max(K, 50)
    blk_wall = timed_wall(blocking_step, n_block, None)

    # ---------------- closed loop with pose feedback (prefetch + localization_fast + mapping)
    def closed_loop(prefetch, depth=False):
        """Whole SLAM step, serial in the pose (src/main.c:300-318): frame t is localised from pose t-1,
        mapped with the fitted pose t.  The prediction is the fitted pose plus the true step."""
        n_steps = max(K, 200)
        spin_up()
        ctx.slam_init(pose_of(0), frames[0], want_global=False)
        out, err, ncorr = NavPos(), C.c_double(0), C.c_size_t(0)
        state = {"last": pose_of(0), "dir": 1}

        def src(cur):
            return (h_depth.data_ptr() + (cur % n_depth) * NPX * 4) if depth else (h_base + cur * FRAME_BYTES)

        def pf(i):
            cur = triangle(i, n_res)
            check((L.nav_slam_prefetch_depth if depth else L.nav_slam_prefetch)(ctx.h, src(cur)))

        def one(i, ahead=True):
            cur, prev = triangle(i, n_res), triangle(i - 1, n_res)
            last = state["last"]
            pred = last + (pose_of(cur) - pose_of(prev)) + np.array([-2.0, 0.5, 0.0, 0.0, 0.0, 0.0])
            pl, pp = pos_c(last), pos_c(pred)
            if prefetch and ahead:
                pf(i + 1)
            check(L.nav_slam_localization_fast(ctx.h, (None if depth else src(cur)) if prefetch else src(cur),
                                               C.byref(pp), C.byref(pl), C.byref(out), C.byref(err), C.byref(ncorr)))
            check(L.nav_slam_mapping(ctx.h, C.byref(out), None, None))
            state["last"] = np.array([out.x, out.y, out.z, out.roll, out.pitch, out.yaw])

        if prefetch:
            pf(1)
        for i in range(1, W + 1):
            one(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(W + 1, W + 1 + n_steps):
            one(i)
        ctx.synchronize()
        barrier()
        wall = reduce_max([time.perf_counter() - t0])[0]
        if prefetch:   # consume the frame prefetched last so that the context is left clean
            one(W + 1 + n_steps, ahead=False)
        ctx.synchronize()
        cur = triangle(W + n_steps + (1 if prefetch else 0), n_res)
        return {"us_per_frame": 1e6 * wall / n_steps, "frames_per_s": world * n_steps / wall, "steps_timed": n_steps,
                "pose_error_mm": float(np.abs(state["last"][:3] - pose_of(cur)[:3]).max()),
                "correspondences": int(ncorr.value), "rms_mm": float(err.value)}

    def closed_loop_c(depth=False):
        """The same loop as ONE C call (nav_slam_run): the prediction is the fitted pose plus a dead-reckoning
        increment per frame, the host loop is the library's, not Python's."""
        n_steps = max(K, 400)
        idx = [triangle(i, n_res) for i in range(0, W + n_steps + 1)]
        bias = np.array([-2.0, 0.5, 0.0, 0.0, 0.0, 0.0])
        deltas = np.stack([pose_of(idx[i]) - pose_of(idx[i - 1]) + bias for i in range(1, len(idx))])
        ptrs = [(h_depth.data_ptr() + (j % n_depth) * NPX * 4) if depth else (h_base + j * FRAME_BYTES) for j in idx[1:]]
        spin_up()
        ctx.slam_init(pose_of(0), frames[0], want_global=False)
        poses, _, _ = ctx.slam_run(ptrs[:W], deltas[:W], pose_of(0), depth_input=depth)
        ctx.synchronize()
        barrier()
        t0 = time.perf_counter()
        poses, errs, ncs = ctx.slam_run(ptrs[W:], deltas[W:], poses[-1], depth_input=depth)
        ctx.synchronize()
        barrier()
        wall = reduce_max([time.perf_counter() - t0])[0]
        return {"us_per_frame": 1e6 * wall / n_steps, "frames_per_s": world * n_steps / wall, "steps_timed": n_steps,
                "api": "nav_slam_run (one C call for the whole timed sequence; upload + labels of frame t+1 under the "
                       "match, fit and mapping of frame t)",
                "h2d_bytes_per_step": NPX * (4 if depth else 24), "d2h_bytes_per_step": 48,
                "pose_error_mm": float(np.abs(poses[-1][:3] - pose_of(idx[-1])[:3]).max()),
                "correspondences": int(ncs[-1]), "rms_mm": float(errs[-1])}

    closed = None
    if not args.skip_closed_loop:
        try:
            closed = {"c_loop": closed_loop_c(), "prefetch": closed_loop(True), "blocking": closed_loop(False)}
            if not args.skip_depth_loop:
                closed["c_loop_depth_input"] = closed_loop_c(depth=True)
                closed["prefetch_depth_input"] = closed_loop(True, depth=True)
        except Exception as ex:  # noqa: BLE001
            closed = {"error": str(ex)[:300]}
    clk = clocks.stop()

    # ---------------- dominant kernel roofline (SURVEY 8d algorithmic bytes)
    torch.cuda.synchronize()
    res = ctx.frame_results_dev()
    nq = int((torch.as_tensor(Raw(res.labels, NPX, "<i4"), device="cuda") == 1).sum())
    n_map = nq  # consecutive frames label ~the same number of points
    n_leaf, n_sup = COLS // 16, COLS // 256
    side = ROWS * (n_leaf * 52 + n_sup * 48)                   # label masks + leaf boxes + super boxes
    alg_bytes = {
        # the single fused frame kernel (labels + match + next map): cloud in, labels + (idx,dist) out,
        # previous map points + masks/boxes in, next global cloud + masks/boxes out
        "frame_fused": NPX * (24 + 4 + 12) + n_map * 24 + side + NPX * 24 + side,
        # transform + map build: cloud + labels in, global cloud out, masks/boxes out
        "map": NPX * (24 + 4 + 24) + side,
    }
    peak, tc_peak, peak_src = measured_peaks()
    seq_mode = window_launches < K          # the library ran the timed steps as one sequence launch
    dom_kernel = "k_frame_seq" if seq_mode else "k_frame_match"
    kernels = {}
    for name, (ms, n) in prof.items():
        if n:
            us = 1e3 * ms / n
            extra = {}
            if name == "frame_fused":
                # the timed region of `value` is K launches of this kernel: its average launch
                # duration there (consecutive launches overlap through programmatic dependent launch) is the
                # step time; the event-bracketed single launch is kept beside it
                extra = {"us_per_launch_isolated": us}
                us, n = 1e3 * dev_ms / K, K
                if seq_mode:
                    # the K timed steps are ONE launch of k_frame_seq (a thread-block cluster per image row walks
                    # through the frames): K frames of algorithmic bytes per launch over that launch's duration
                    extra.update({"frames_per_launch": K, "us_per_frame": us})
                    us, n = 1e3 * dev_ms, 1
            ab = alg_bytes[name] * (K if (seq_mode and name == "frame_fused") else 1)
            ach = ab / (us * 1e-6) / 1e9
            kernels[name] = {"us_per_launch": us, "launches": n, "alg_bytes_per_launch": ab,
                             "achieved_gbs": ach, "frac_of_hbm_peak": ach / peak, **extra}
    dom = "frame_fused" if "frame_fused" in kernels else (max(kernels, key=lambda k: kernels[k]["us_per_launch"]) if kernels else None)
    # DRAM traffic of the dominant kernel: from the committed ncu --set full capture of this round (a live
    # counter read needs a profiler, and a number taken under a profiler is never a bench value)
    traffic, traffic_src = None, None
    for cand in ("r2_traffic.json", "r1_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", cand)) as f:
                tk = json.load(f)["kernels"]
            for name, v in tk.items():
                if dom_kernel in name:
                    traffic = v["dram_read_bytes"] + v["dram_write_bytes"]
                    if seq_mode:   # captured with frames_per_launch frames in the launch: scale to this run's K
                        traffic = traffic * K / v.get("frames_per_launch", K)
                    traffic_src = f"profiles/{cand}"
            if traffic is not None:
                break
        except (OSError, KeyError, ValueError):
            continue

    # ---------------- the stencil on a device-resident batch (north_star: >= 60 % of HBM peak)
    # a buffer of its own, sized by --stencil-images (default 512 = 1.6 GB of input, 13x the L2), whatever --steps is
    n_b = args.stencil_images
    reps_idx = torch.arange(n_b, device="cuda") % n_res
    d_batch = d_frames.index_select(0, reps_idx)
    d_lab = torch.empty((n_b, ROWS, COLS), dtype=torch.int32, device="cuda")
    spin_up()
    for _ in range(3):
        ctx.extract_feature_batch_dev(d_batch.data_ptr(), n_b, d_lab.data_ptr())
    st = []
    for _ in range(7):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ctx.extract_feature_batch_dev(d_batch.data_ptr(), n_b, d_lab.data_ptr())
        e1.record(stream)
        st.append((e0, e1))
    torch.cuda.synchronize()
    st_ms = float(np.median([a.elapsed_time(b) for a, b in st]))
    st_bytes = n_b * NPX * 28
    kernels["labels_batch"] = {"kernel": "k_labels_tma", "images": n_b, "us_per_launch": 1e3 * st_ms,
                               "alg_bytes_per_launch": st_bytes,
                               "achieved_gbs": st_bytes / (st_ms * 1e-3) / 1e9,
                               "frac_of_hbm_peak": st_bytes / (st_ms * 1e-3) / 1e9 / peak,
                               "input_bytes": n_b * FRAME_BYTES,
                               "note": "dedicated batch buffer, %.2f GB in + %.2f GB out per launch (L2 is 0.13 GB), "
                                       "median of 7 launches" % (n_b * FRAME_BYTES / 1e9, n_b * NPX * 4 / 1e9)}
    del d_batch, d_lab

    # ---------------- config 5a: 8 independent sequences spread over the ranks (8 / world per rank, side by side
    # in every launch)
    batched = None
    if not args.skip_batched:
        S = max(1, 8 // world)
        Fb = min(n_res // S, 33)
        ctx8 = pkg.Context(ROWS, COLS, device=local, n_seq=S)
        ctx8.set_stream(stream.cuda_stream)
        # sequence s uses frames s, s+S, s+2S ... of the resident set (distinct data per sequence)
        d8 = d_frames[: S * Fb].reshape(Fb, S, ROWS, COLS, 3)
        pp = np.stack([np.stack([poses_for(f + 1)[0]] * S) for f in range(Fb)])
        pl = np.stack([np.stack([poses_for(f + 1)[1]] * S) for f in range(Fb)])
        pf = np.stack([np.stack([poses_for(f + 1)[2]] * S) for f in range(Fb)])
        spin_up()
        ctx8.slam_init_dev(d8[0].data_ptr(), pf[0])
        ctx8.frontend_sequence_dev(d8[1].data_ptr(), Fb - 1, pp[1:], pl[1:], pf[1:])
        barrier()
        bms = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ctx8.slam_init_dev(d8[0].data_ptr(), pf[0])
            e0.record(stream)
            ctx8.frontend_sequence_dev(d8[1].data_ptr(), Fb - 1, pp[1:], pl[1:], pf[1:])
            e1.record(stream)
            bms.append((e0, e1))
        barrier()
        b_ms = reduce_max([float(np.median([a.elapsed_time(b) for a, b in bms]))])[0]
        batched = {"workload": "cfg5a: 8 independent 64x2048 sequences over %d GPU(s), %d per rank side by side in "
                               "every launch" % (world, S),
                   "n_seq_per_rank": S, "frames": world * S * (Fb - 1), "ms": b_ms,
                   "frames_per_s": world * S * (Fb - 1) / (b_ms * 1e-3)}
        ctx8.close()

    # ---------------- kd-tree path: config 4 (1 M-point map) at N=1, config 5b (10 M-point map, queries sharded
    # across ranks against a replicated tree, one all_gather) at N>1
    nn = None
    if not args.skip_kdtree:
        nn = kd_legs(args, torch, dist, pkg, stream, world, rank, local, spin_up, barrier, reduce_max, peak, tc_peak)

    shim = None
    if rank == 0 and world == 1 and not args.skip_shim:
        ctx.synchronize()
        shim = shim_legs()
        if cpu and cpu.get("whole_step_ms_per_frame"):
            shim["reference_whole_step_ms_per_frame"] = cpu["whole_step_ms_per_frame"]

    if rank == 0:
        value = world * K / (dev_ms * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "frames_resident": n_res, "frame_bytes": FRAME_BYTES,
                       "l2_policy": "inputs larger than L2: every step reads a different 3.1 MB frame of a %.2f GB "
                                    "resident sequence (L2 is 0.13 GB); the previous frame's row map (5 MB) is "
                                    "legitimately L2-warm; the clock spin-up between regions runs on a buffer of its own"
                                    % (n_res * FRAME_BYTES / 1e9),
                       "timing": "the K = %d timed steps (frames %d..%d) between one pair of CUDA events, after 3 untimed "
                                 "passes over the same frames and %d untimed warm-up steps; ms_per_step = that time / K, "
                                 "MAX over ranks" % (K, F0 + W, F0 + W + K - 1, W)},
            "timed_region": {"steps": K, "device_ms": dev_ms, "launches": window_launches,
                             "ms_per_step_per_rank": per_rank},
            # headline e2e: pinned cloud in, the step's results (labels as bit masks + NN index + NN distance) out,
            # per frame, pipelined.  The mapped global cloud is persistent state (the next frame's search structure
            # and the source of the GPU CSV writer) and stays in HBM; the other variants are reported beside it.
            "e2e": {**e2e_masks,
                    "api": "nav_frontend_submit(cloud, mask_out, nn_idx_out, nn_dist_out) + nav_frontend_wait (pinned host "
                           "buffers; upload, kernels and download of consecutive frames overlap on three streams)",
                    "h2d_bytes_per_step": FRAME_BYTES,
                    "d2h_bytes_per_step": NPX * 12 + ROWS * n_chunks * 4,
                    "int_labels": {**e2e_labels, "api": "same call with feature_out (int labels, 512 KB) instead of mask_out",
                                   "h2d_bytes_per_step": FRAME_BYTES, "d2h_bytes_per_step": NPX * 16},
                    "with_global_cloud": {**e2e_all, "api": "same, global_out given too: the 3.1 MB mapped cloud is downloaded",
                                          "h2d_bytes_per_step": FRAME_BYTES, "d2h_bytes_per_step": NPX * 40},
                    "depth_input": {**e2e_depth,
                                    "api": "nav_frontend_submit(distances, mask_out, nn_idx_out, nn_dist_out): L5-type depth "
                                           "matrix in (utils/pointcloud.c:8 runs on the device)",
                                    "h2d_bytes_per_step": NPX * 4, "d2h_bytes_per_step": NPX * 12 + ROWS * n_chunks * 4},
                    "depth_input_idx_only": {**e2e_depth_idx,
                                             "api": "same with nn_dist_out = NULL: label masks + NN indices come back (the "
                                                    "smallest per-pixel result; what still scales when eight ranks share the "
                                                    "host's PCIe fabric)",
                                             "h2d_bytes_per_step": NPX * 4, "d2h_bytes_per_step": NPX * 4 + ROWS * n_chunks * 4},
                    "blocking_call": {"value": world * n_block / blk_wall, "unit": "frames/s",
                                      "api": "nav_frontend_frame (all four outputs, returns with the results on the host)",
                                      "wall_ms_per_step": 1e3 * blk_wall / n_block}},
            "e2e_closed_loop": closed, "e2e_shim": shim,
            "gpu_launches": 1 if seq_mode else int(round(K)),
            "gpu_launches_note": ("ONE launch of k_frame_seq covers the K timed steps (a thread-block cluster "
                                  "per image row walks through the frames; %.0f launches in the window including the untimed "
                                  "re-init and warm-up; NAV_SEQ_LAUNCHES=1 gives one k_frame_match launch per step)"
                                  if seq_mode else
                                  "K launches of k_frame_match in the timed region (%.0f launches in the window including the "
                                  "untimed re-init and warm-up)") % window_launches,
            "clocks": clk, "cpu_cores_bound_near_gpu": bound_cores,
            "roofline": None if dom is None else {
                "kernel": {"frame_fused": ("k_frame_seq (labels + match + next map, K frames per launch)" if seq_mode else
                                           "k_frame_match<fused labels, fused map>")}.get(dom, dom), "bound": "hbm",
                "achieved": kernels[dom]["achieved_gbs"], "peak": peak,
                "peak_source": peak_src, "unit": "GB/s", "frac": kernels[dom]["frac_of_hbm_peak"], "traffic": traffic,
                "traffic_source": traffic_src,
                "alg_bytes_per_launch": kernels[dom]["alg_bytes_per_launch"],
                "us_per_launch": kernels[dom]["us_per_launch"],
                "note": "3 MB per frame and a serial dependency from frame to frame: bounded by instruction issue and the "
                        "latency chain of one image row, not by HBM; "
                        "the same stencil fed a batch reaches kernels.labels_batch.frac_of_hbm_peak"},
            "kernels": kernels, "batched_sequences": batched, "nn": nn, "cpu_baseline": cpu,
        }
        print_line(line)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def kd_legs(args, torch, dist, pkg, stream, world, rank, local, spin_up, barrier, reduce_max, peak, tc_peak):
    sharding = importlib.import_module("nav-slam_b200.sharding")
    n_map = 10_000_000 if (world > 1 or args.big_map) else 1_000_000
    nq = 131072
    s = stream.cuda_stream
    d_pts = torch.empty((n_map, 3), dtype=torch.float64, device="cuda")
    if rank == 0:
        d_pts.copy_(torch.from_numpy(pkg.synth.map_points(n_map)))
    sharding.broadcast_points(d_pts)                                   # NCCL broadcast (no-op at N=1)
    sample = d_pts[:: max(n_map // 200000, 1)].cpu().numpy()          # queries derive from the map
    d_q = torch.from_numpy(pkg.synth.map_queries(sample, nq)).cuda()

    def time_build(ptr, n, reps=5):
        pkg.KdTree(dev_ptr=ptr, n=n, device=local, stream=s).close()   # warm the allocator
        spin_up()
        ts, tree = [], None
        for _ in range(reps):
            if tree is not None:
                tree.close()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            tree = pkg.KdTree(dev_ptr=ptr, n=n, device=local, stream=s)
            e1.record(stream)
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return tree, float(np.median(ts)), int(tree.launch_count())

    tree, b_ms, b_launches = time_build(d_pts.data_ptr(), n_map)
    buf_i = torch.empty(nq, dtype=torch.int32, device="cuda")
    buf_d = torch.empty(nq, dtype=torch.float64, device="cuda")

    def nn_into(qs, idx_view, dist_view):   # this rank's shard of the queries, answers written in place
        tree.nn_batch_dev(qs.data_ptr(), int(qs.shape[0]), idx_view.data_ptr(), dist_view.data_ptr(), s)

    def time_steps(fn, reps=10):
        spin_up()
        for _ in range(3):
            fn()
        barrier()
        evs = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            evs.append((e0, e1))
        barrier()
        return float(np.median([a.elapsed_time(b) for a, b in evs]))

    q_ms = time_steps(lambda: sharding.sharded_nn_into(nn_into, d_q, buf_i, buf_d))
    matched = int((buf_i >= 0).sum())
    q_ms, b_ms = reduce_max([q_ms, b_ms])
    # the same exchange over peer memory: the search kernel stores its shard's answers into the buffers of all ranks
    # (CUDA IPC mappings, NVLink stores) and no collective follows (nav_kdtree_nn_allgather_dev)
    peer, peer_ms, peer_same, peer_err = None, None, None, None
    if world > 1:
        try:
            peer = sharding.PeerGather(pkg.load_library(), local, nq * world)   # sized for the weak-scaling run too
            peer.nq = nq
            pi, pd = peer.nn(tree, d_q, s)
            torch.cuda.synchronize()
            peer_same = bool(torch.equal(pi[:nq], buf_i) and torch.equal(pd[:nq], buf_d))
            peer_ms = reduce_max([time_steps(lambda: peer.nn(tree, d_q, s))])[0]
            peer.check()
        except Exception as ex:  # noqa: BLE001
            peer_err = str(ex)[:200]
            if peer is not None:
                peer.close()
            peer = None
    ag_ms = q_ms
    if peer_ms is not None:      # the headline of 5b is the exchange over peer memory; the all_gather stays beside it
        q_ms = peer_ms
    nn = {"workload": (("cfg5b: 10 M-point map replicated, 131072 queries sharded over %d ranks, " % world) +
                       ("answers stored into every rank's buffer by the search kernel (peer memory over NVLink)"
                        if peer_ms is not None else "one packed all_gather"))
          if world > 1 else ("cfg4: %d-point map, 131072 queries" % n_map),
          "all_gather_query_ms": ag_ms if world > 1 else None,
          "map_points": n_map, "queries": nq, "build_ms": b_ms, "build_launches": b_launches, "query_ms": q_ms,
          "queries_per_s": nq / (q_ms * 1e-3), "matched": matched,
          "peer_memory": None if world == 1 else (
              {"error": peer_err} if peer_ms is None else
              {"exchange": "no collective: the search kernel stores its shard's answers into every rank's buffer over "
                           "NVLink (CUDA IPC mappings) and posts a flag; a one-warp kernel waits for the flags",
               "query_ms": peer_ms, "queries_per_s": nq / (peer_ms * 1e-3), "same_answers_as_all_gather": peer_same}),
          "roofline_query": {"kernel": "k_kd_nn_stack", "bound": "hbm (latency-bound traversal; tree bytes are cache traffic)",
                             "alg_bytes_per_launch": nq * 36 // world, "achieved": nq * 36 / (q_ms * 1e-3) / 1e9,
                             "peak": peak, "unit": "GB/s", "frac": nq * 36 / (q_ms * 1e-3) / 1e9 / peak},
          # SURVEY 8d: the build's lower bound is 24 B read + 32 B node written per point
          "roofline_build": {"kernel": "kd_build (all launches of one build)", "bound": "hbm",
                             "alg_bytes": n_map * 56, "achieved": n_map * 56 / (b_ms * 1e-3) / 1e9, "peak": peak,
                             "unit": "GB/s", "frac": n_map * 56 / (b_ms * 1e-3) / 1e9 / peak}}
    if world > 1:
        # weak-scaling variant: 131072 queries PER RANK (the exchange grows with the world, the search does not)
        nq_w = nq * world
        d_qw = torch.from_numpy(pkg.synth.map_queries(sample, nq_w, seed=4002)).cuda()
        wi = torch.empty(nq_w, dtype=torch.int32, device="cuda")
        wd = torch.empty(nq_w, dtype=torch.float64, device="cuda")
        w_ms = reduce_max([time_steps(lambda: sharding.sharded_nn_into(nn_into, d_qw, wi, wd))])[0]
        nn["weak_scaling"] = {"queries_total": nq_w, "queries_per_rank": nq, "query_ms": w_ms,
                              "queries_per_s": nq_w / (w_ms * 1e-3)}
        if peer is not None:
            try:
                peer.nq = nq_w
                wp_ms = reduce_max([time_steps(lambda: peer.nn(tree, d_qw, s))])[0]
                peer.check()
                nn["weak_scaling"]["peer_memory_query_ms"] = wp_ms
                nn["weak_scaling"]["peer_memory_queries_per_s"] = nq_w / (wp_ms * 1e-3)
            except Exception as ex:  # noqa: BLE001
                nn["weak_scaling"]["peer_memory_error"] = str(ex)[:200]
        del d_qw, wi, wd
    if peer is not None:
        # the MAP sharded instead of the queries: every rank builds 1/world of the points and searches it for all
        # queries; partial answers meet at the owners of the queries, merged answers go to everybody (two rounds over
        # peer memory).  What a map that is rebuilt every frame wants: the build shrinks with the world.
        try:
            peer.nq = nq
            lo_p, hi_p = sharding.shard_bounds(n_map, world, rank)
            part, pb_ms, pb_launches = time_build(d_pts[lo_p:hi_p].data_ptr(), hi_p - lo_p)
            si, sd = peer.nn_sharded_map(part, d_q, lo_p, s)
            torch.cuda.synchronize()
            same = bool(torch.equal(si[:nq], buf_i) and torch.equal(sd[:nq], buf_d))
            sm_ms = time_steps(lambda: peer.nn_sharded_map(part, d_q, lo_p, s))
            peer.check()
            sm_ms, pb_ms = reduce_max([sm_ms, pb_ms])
            nn["sharded_map"] = {
                "workload": "cfg5b with the MAP sharded: %d ranks x %d points, all 131072 queries on every rank, partial "
                            "answers merged by the owners of the queries over peer memory" % (world, hi_p - lo_p),
                "build_ms": pb_ms, "build_launches": pb_launches, "query_ms": sm_ms, "queries_per_s": nq / (sm_ms * 1e-3),
                "same_answers_as_replicated_tree": same,
                "build_plus_query_ms": pb_ms + sm_ms, "replicated_build_plus_query_ms": b_ms + (peer_ms or q_ms)}
            part.close()
        except Exception as ex:  # noqa: BLE001
            nn["sharded_map"] = {"error": str(ex)[:200]}
        barrier()
        peer.close()
    tree.close()
    del d_pts
    if world == 1 and not args.big_map:
        # config 4 the way a SLAM run produces it: 8 mapped 64x2048 frames (1 048 576 points lying on
        # the room's surfaces) queried by the next frame's 131 072 points in image order
        pts_a, q_a = pkg.synth.accumulated_map(8)
        d_pa, d_qa = torch.from_numpy(pts_a).cuda(), torch.from_numpy(q_a).cuda()
        tree, ba_ms, _ = time_build(d_pa.data_ptr(), pts_a.shape[0])
        qa_ms = time_steps(lambda: tree.nn_batch_dev(d_qa.data_ptr(), nq, buf_i.data_ptr(), buf_d.data_ptr(), s))
        nn["accumulated_map"] = {
            "workload": "cfg4 as a SLAM run produces it: 8 mapped 64x2048 room frames (surfaces), queried by the "
                        "next frame's points in image order",
            "map_points": int(pts_a.shape[0]), "queries": nq, "build_ms": ba_ms, "query_ms": qa_ms,
            "queries_per_s": nq / (qa_ms * 1e-3), "matched": int((buf_i >= 0).sum())}
        kd_idx = buf_i.clone()
        kd_dist = buf_d.clone()
        tree.close()
        if not args.skip_tc:
            # config 4, second half: the tensor-core brute force on the same 1 M x 131 072 problem (same answers)
            try:
                tc_i = torch.empty(nq, dtype=torch.int32, device="cuda")
                tc_d = torch.empty(nq, dtype=torch.float64, device="cuda")

                def tc():
                    pkg.bruteforce_nn_dev(local, d_pa.data_ptr(), int(pts_a.shape[0]), d_qa.data_ptr(), nq, tc_i.data_ptr(),
                                          tc_d.data_ptr(), use_tensor_cores=True, stream=s)
                tc_ms = time_steps(tc, reps=3)
                flop = 2.0 * nq * pts_a.shape[0] * 32 * 2    # two passes over K = 32 bf16 products
                nn["tensor_core_bruteforce"] = {
                    "workload": "cfg4: the same accumulated 1 M-point map and 131072 queries, tcgen05 candidate tiles + exact "
                                "binary64 re-rank (nav_bruteforce_nn_batch_dev, use_tensor_cores = 1)",
                    "ms": tc_ms, "queries_per_s": nq / (tc_ms * 1e-3),
                    "same_answers_as_kdtree": bool(torch.equal(tc_i, kd_idx) and torch.equal(tc_d, kd_dist)),
                    "kdtree_ms": qa_ms, "kdtree_build_ms": ba_ms,
                    "roofline": {"bound": "tensor", "achieved": flop / (tc_ms * 1e-3) / 1e12, "peak": tc_peak,
                                 "unit": "TFLOP/s", "frac": flop / (tc_ms * 1e-3) / 1e12 / tc_peak,
                                 "note": "bf16 flops of both tile passes (K = 32) over the whole call, re-rank included"}}
            except Exception as ex:  # noqa: BLE001
                nn["tensor_core_bruteforce"] = {"error": str(ex)[:300]}
        del d_pa, d_qa
    return nn


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=256, help="frames of the resident sequence (805 MB at 256)")
    ap.add_argument("--min-timed-ms", type=float, default=60.0, help="device time to accumulate in the e2e legs")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the results of the last timed step (rank 0) as DIR/<name>.npy")
    ap.add_argument("--stencil-images", type=int, default=512)
    ap.add_argument("--cpu-frames", type=int, default=60)
    ap.add_argument("--cpu-whole-frames", type=int, default=3)
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-kdtree", action="store_true")
    ap.add_argument("--skip-batched", action="store_true")
    ap.add_argument("--skip-closed-loop", action="store_true")
    ap.add_argument("--skip-depth-loop", action="store_true")
    ap.add_argument("--skip-shim", action="store_true")
    ap.add_argument("--skip-tc", action="store_true")
    ap.add_argument("--big-map", action="store_true", help="use the 10 M-point map at N=1 too")
    ap.add_argument("--shim-leg", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--shim-out", default="", help=argparse.SUPPRESS)
    ap.add_argument("--shim-frames", type=int, default=20, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.shim_leg:
        run_shim_leg(args)
        return
    # stdout carries the ONE JSON line and nothing else: libraries that write to file descriptor 1 (NCCL prints
    # its version there) are sent to stderr, and print_line() writes the line to the real stdout
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
