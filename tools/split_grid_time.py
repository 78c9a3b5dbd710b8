#!/usr/bin/env python
"""Experiment (not a test): where the split kernel's time goes on few CTAs per frame (the frame pipeline's case).

On the 32 bench frames (G1 3840x2160, seeds 12345..12376, K = 256), through dq_quant_recurse_device:
  1. the split stage alone (dq_context_set_profiling -> stage_ms["split"]) at each grid size of --ctas:
     median and range over every frame and repetition, plus a digest of all palettes and outputs (the results do not
     depend on the grid, and two builds must print the same digest);
  2. at --trace-ctas CTAs, CTA 0's timeline (dq_debug_split_timeline) per round, averaged over the frames:
     controller (phases a-c), wide passes, wide partition, narrow jobs, grid barrier; the round's jobs, CTA 0's wide /
     narrow jobs, its wide passes and (when the build records them, tag 13) the passes each narrow job ran.
Cycles become microseconds through each call's own split time (timeline span / stage_ms["split"]).

usage: python tools/split_grid_time.py [--ctas 4,8,12,148] [--reps 3] [--trace-ctas 8]
A/B of two builds: DIVQUANT_B200_LIB=<other libdivquant_b200.so> python tools/split_grid_time.py"""
import argparse
import ctypes as C
import hashlib
import importlib
import os
import statistics
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import Oracle  # noqa: E402  (input generator only)

W, H, K = 3840, 2160, 256
SEEDS = list(range(12345, 12345 + 32))
TAGS = {1: "round", 2: "phaseA", 3: "phaseB", 4: "phaseC", 5: "ctlbar", 6: "pass", 7: "part", 8: "root", 9: "begin",
        10: "collected", 11: "reduced", 12: "rootbar", 13: "narrow_job"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ctas", default="4,8,12,148")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--trace-ctas", type=int, default=8)
    args = ap.parse_args()
    pkg = importlib.import_module("clusteringsegmentation-1_b200")
    lib = pkg.load_library()
    lib.dq_set_display_timings(0)
    print("library:", os.path.relpath(os.environ.get("DIVQUANT_B200_LIB", pkg.LIB_PATH), ROOT), "| device:", torch.cuda.get_device_name(0),
          flush=True)
    o = Oracle()
    frames = [torch.from_numpy(o.generate(1, W, H, s).view(np.int32)).cuda() for s in SEEDS]
    out = torch.empty_like(frames[0])
    ctx = lib.dq_context_create(0)
    lib.dq_context_set_profiling(ctx, 1)
    ct = (C.c_uint32 * K)()
    nk = C.c_uint32(K)
    st = pkg.CallStats()

    def call(f):
        nk.value = K
        lib.dq_quant_recurse_device(ctx, frames[f].numel(), frames[f].data_ptr(), out.data_ptr(), C.byref(nk), ct, 0)
        lib.dq_context_last_stats(ctx, C.byref(st))
        return st.as_dict()

    for g in (int(x) for x in args.ctas.split(",")):
        lib.dq_context_set_split_ctas(ctx, g)
        digest = hashlib.sha256()
        for f in range(len(frames)):  # warm-up, and the digest of every result
            call(f)
            torch.cuda.synchronize()
            digest.update(bytes(ct)[: 4 * nk.value])
            digest.update(out.cpu().numpy().tobytes())
        ms = []
        for _ in range(args.reps):
            for f in range(len(frames)):
                ms.append(call(f)["stage_ms"]["split"])
        print(f"split_ctas={g:3d}: split stage median {statistics.median(ms):.4f} ms, range {min(ms):.4f}-{max(ms):.4f} "
              f"({len(ms)} calls), results sha256 {digest.hexdigest()[:16]}", flush=True)

    # ---- CTA 0's timeline, per round ----
    g = args.trace_ctas
    lib.dq_context_set_split_ctas(ctx, g)
    buf = (C.c_uint64 * 8192)()
    rounds = {}  # round -> {phase: [us per frame]}
    narrow_passes = []
    totals = []
    for f in range(len(frames)):
        lib.dq_debug_split_timeline(ctx, 1, None, 0)
        d = call(f)
        torch.cuda.synchronize()
        n = lib.dq_debug_split_timeline(ctx, 0, buf, 4096)
        lib.dq_debug_split_timeline(ctx, 0, None, 0)
        ev = [(int(buf[2 * i] >> 32), int(buf[2 * i] & 0xFFFFFFFF), int(buf[2 * i + 1])) for i in range(n)]
        if not ev:
            print("no timeline recorded", flush=True)
            return
        us_per_cycle = d["stage_ms"]["split"] * 1e3 / max(ev[-1][2] - ev[0][2], 1)
        totals.append((ev[-1][2] - ev[0][2]) * us_per_cycle)
        cur, last, r = None, ev[0][2], -1
        for tag, arg, clk in ev:
            dt = (clk - last) * us_per_cycle
            last = clk
            name = TAGS.get(tag, str(tag))
            if name == "round":
                r = arg
                cur = rounds.setdefault(r, {})
                cur.setdefault("frames", 0)
                cur["frames"] += 1
                cur["controller"] = cur.get("controller", 0.0) + dt  # cta_error() after the previous barrier
                continue
            if cur is None:
                phase = "root"
            elif name in ("phaseA", "phaseB", "phaseC"):
                phase = "controller"
                if name == "phaseC":
                    cur["jobs"] = cur.get("jobs", 0) + arg
            elif name == "pass":
                phase = "wide_passes"
                cur["cta0_wide_passes"] = cur.get("cta0_wide_passes", 0) + 1
            elif name == "narrow_job":
                phase = "narrow"
                narrow_passes.append(arg)
                cur.setdefault("passes", []).append(arg)
            elif name == "part" and arg < 1000:
                phase = "wide_partition"
                cur["cta0_wide_jobs"] = cur.get("cta0_wide_jobs", 0) + arg
            elif name == "part":
                phase = "narrow"
                cur["cta0_narrow_jobs"] = cur.get("cta0_narrow_jobs", 0) + arg - 1000
            elif name == "ctlbar":
                phase = "barrier"
            else:
                phase = name
            if cur is not None:
                cur[phase] = cur.get(phase, 0.0) + dt
    nf = len(frames)
    print(f"\nCTA 0 timeline at split_ctas={g}, mean over {nf} frames (us; the split stage spans {statistics.mean(totals):.1f} us):")
    cols = ("controller", "wide_passes", "wide_partition", "narrow", "barrier")
    print(f"{'round':>5} {'frames':>6} {'jobs':>6} {'w/CTA0':>6} {'n/CTA0':>6} {'wpass':>5} " + " ".join(f"{c:>14}" for c in cols)
          + "   narrow passes (mean, CTA 0)")
    tot = dict.fromkeys(cols, 0.0)
    for r in sorted(rounds):
        x = rounds[r]
        fr = x["frames"]
        p = x.get("passes", [])
        line = (f"{r:5d} {fr:6d} {x.get('jobs', 0) / fr:6.1f} {x.get('cta0_wide_jobs', 0) / fr:6.1f} "
                f"{x.get('cta0_narrow_jobs', 0) / fr:6.1f} {x.get('cta0_wide_passes', 0) / fr:5.1f} ")
        line += " ".join(f"{x.get(c, 0.0) / nf:14.1f}" for c in cols)
        line += f"   {statistics.mean(p):.2f}" if p else "   -"
        print(line)
        for c in cols:
            tot[c] += x.get(c, 0.0) / nf
    print("total " + " ".join(f"{c}={v:.1f}" for c, v in tot.items()) + f"  sum={sum(tot.values()):.1f} us")
    if narrow_passes:
        hist = np.bincount(np.array(narrow_passes), minlength=12)
        print("passes per narrow job on CTA 0 (1 cut pass + LKM passes, final included):",
              {i: int(c) for i, c in enumerate(hist) if c}, f"mean {np.mean(narrow_passes):.2f}")
    else:
        print("passes per narrow job: not recorded by this build (no tag 13)")
    lib.dq_context_destroy(ctx)


if __name__ == "__main__":
    main()
