#!/usr/bin/env python
"""Cost of the reference tie rule (Context.set_tie_rule("reference"), NAV_TIE_REFERENCE) against the default
lowest-index rule, on the blocking calls that support it, at 16x1800 (integer-mm L9 frames, synth.l9_sequence: exact
distance ties in every frame) and 64x2048 (fp64 room frames, synth.room_sequence: no ties).

Per shape and rule: host wall-clock time per call of slam_match, slam_localization and frontend_frame (every such call
ends in a stream synchronisation), each over the same FRAMES frames after a warm-up pass, rules alternating, ROUNDS
rounds (the median is printed); the number of queries the host resolved per frame; and, in a separate profiled pass
(nav_profile_enable), the split of the reference rule's overhead into the match kernel's extra device time (CUDA
events), the copies of the tie list and rows to the host, the host's tree builds and searches, and the upload of the
answers with the scatter launch.  The card's name and power limit are read in the same run.
usage: prof_ref_ties.py [out_path]"""
import importlib
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
nav = importlib.import_module("nav-slam_b200")

OUT = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_ref_ties.txt")
FRAMES, ROUNDS = 20, 3
STEP = np.array([48.0, 1.0, 0.0, 0.0, 0.0, 0.0])
RULES = ("lowest_index", "reference")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


def workload(shape):
    r, c = shape
    if shape == (16, 1800):
        return nav.synth.l9_sequence(FRAMES + 1)
    return nav.synth.room_sequence(r, c, FRAMES + 1)


def run_calls(ctx, frames, call):
    """one pass over the frames; returns (seconds per call, resolved queries per frame)"""
    ctx.slam_init(np.zeros(6), frames[0], want_global=False)
    last = np.zeros(6)
    r0 = ctx.tie_resolve_count()
    t = 0.0
    for f in range(1, len(frames)):
        pred = last + STEP
        t0 = time.perf_counter()
        if call == "slam_match":
            ctx.slam_match(frames[f], pred, last)
        elif call == "slam_localization":
            ctx.slam_localization(frames[f], pred, last)
        else:
            ctx.frontend_frame(frames[f], pred, last, pred)
        t += time.perf_counter() - t0
        if call != "frontend_frame":
            ctx.slam_mapping(pred, frames[f], want_global=False)
        last = pred
    n = len(frames) - 1
    return t / n, (ctx.tie_resolve_count() - r0) / n


def main():
    lines = [f"# profiles/prof_ref_ties.py -- {gpu_info()} (name, power limit, max SM clock)",
             f"# {FRAMES} frames per pass, {ROUNDS} rounds, rules alternating; host wall clock per blocking call, median "
             f"of the rounds"]
    for shape in ((16, 1800), (64, 2048)):
        frames = workload(shape)
        ctxs = {}
        for rule in RULES:
            ctxs[rule] = nav.Context(*shape)
            ctxs[rule].set_tie_rule(rule)
        lines.append(f"\n## {shape[0]}x{shape[1]} ({'integer-mm L9' if shape == (16, 1800) else 'fp64 room'} frames)")
        lines.append(f"{'call':<18} {'rule':<13} {'us/call':>10} {'flagged/frame':>14}")
        for call in ("slam_match", "slam_localization", "frontend_frame"):
            for rule in RULES:  # warm-up
                run_calls(ctxs[rule], frames[:3], call)
            res = {rule: [] for rule in RULES}
            for _ in range(ROUNDS):
                for rule in RULES:
                    res[rule].append(run_calls(ctxs[rule], frames, call))
            for rule in RULES:
                t = float(np.median([v[0] for v in res[rule]]))
                lines.append(f"{call:<18} {rule:<13} {t * 1e6:10.1f} {res[rule][0][1]:14.1f}")
        # overhead split of the reference rule, profiled pass (frontend_frame and slam_match)
        lines.append("overhead split (profiled pass, per call): match kernel device time by rule; host ms of the tie "
                     "steps under the reference rule")
        for call in ("slam_match", "frontend_frame"):
            km = {}
            for rule in RULES:
                ctx = ctxs[rule]
                ctx.profile_enable(True)
                for name in ("match", "tie_copies", "tie_search", "tie_upload"):
                    ctx.profile_read(name, reset=True)
                run_calls(ctx, frames, call)
                ms, n = ctx.profile_read("match", reset=True)
                km[rule] = 1e3 * ms / max(n, 1)
                if rule == "reference":
                    steps = {name: ctx.profile_read(name, reset=True) for name in ("tie_copies", "tie_search", "tie_upload")}
                ctx.profile_enable(False)
            per = {k: 1e3 * v[0] / FRAMES for k, v in steps.items()}
            lines.append(f"  {call:<16} match kernel {km['lowest_index']:.1f} us (lowest_index) vs {km['reference']:.1f} "
                         f"us (reference): {km['reference'] - km['lowest_index']:+.1f} us; copies {per['tie_copies']:.1f} "
                         f"us, host trees+searches {per['tie_search']:.1f} us, upload+scatter {per['tie_upload']:.1f} us "
                         f"(frames with ties: {steps['tie_upload'][1]} of {FRAMES})")
        for ctx in ctxs.values():
            ctx.close()
    text = "\n".join(lines) + "\n"
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    with open(OUT, "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    main()
