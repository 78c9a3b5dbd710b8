#!/usr/bin/env python
"""Experiment (not a test): where a frame's time goes inside the frame pipeline.  Runs device-resident G1 frames through
`lanes` lanes under torch.profiler (CUDA activities) and prints, per kernel family, how many launches it saw and their
mean / total duration.  The kernels of different lanes overlap, so these are durations inside the pipeline, not shares of
its wall time; run it on its own (the profiler slows the host) and take throughput from tools/lanes_check.py.
usage: python tools/pipe_trace.py [width height K frames lanes [trace.json]]"""
import ctypes as C
import importlib
import os
import sys
from collections import defaultdict

import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import Oracle  # input generator only  # noqa: E402

args = sys.argv[1:]
w, h, k, frames, lanes = [int(x) for x in (args[:5] + ["3840", "2160", "256", "96", "12"][len(args[:5]):])]
trace_path = args[5] if len(args) > 5 else None
FAMILIES = ("hist_insert", "map_gather", "map_unique", "split2_kernel")

pkg = importlib.import_module("clusteringsegmentation-1_b200")
lib = pkg.load_library()
lib.dq_set_display_timings(0)
n = w * h
o = Oracle()
dev = [torch.from_numpy(o.generate(1, w, h, 12345 + s).view(np.int32)).cuda() for s in range(min(frames, 8))]
nbuf = lanes + 2
outs = [torch.empty(n, dtype=torch.int32, device="cuda") for _ in range(nbuf)]
pipe = lib.dq_pipeline_create_lanes(0, 0, lanes, 0)
u32p = C.POINTER(C.c_uint32)


def run(count):
    nks = [C.c_uint32(k) for _ in range(count)]
    cts = [np.zeros(k, np.uint32) for _ in range(count)]
    tickets = []
    for i in range(count):
        if len(tickets) >= nbuf:  # the out buffer about to be reused must be complete
            lib.dq_pipeline_wait(pipe, tickets[i - nbuf])
        tickets.append(lib.dq_pipeline_submit_device(pipe, n, dev[i % len(dev)].data_ptr(), outs[i % nbuf].data_ptr(),
                                                     C.byref(nks[i]), cts[i].ctypes.data_as(u32p), 0))
    lib.dq_pipeline_flush(pipe)


run(2 * lanes)  # warm-up: modules, lane buffers
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    run(frames)
    torch.cuda.synchronize()
ms_frame = lib.dq_pipeline_last_elapsed_ms(pipe) / frames
lib.dq_pipeline_destroy(pipe)
if trace_path:
    prof.export_chrome_trace(trace_path)

stats = defaultdict(list)
for ev in prof.events():
    if ev.device_type != torch.autograd.DeviceType.CUDA:
        continue
    for fam in FAMILIES:
        if fam in ev.name:
            stats[fam].append(ev.time_range.elapsed_us())
print(f"{w}x{h} K={k}, {frames} frames, {lanes} lanes: {ms_frame:.3f} ms/frame (pipeline events, under the profiler)")
for fam in FAMILIES:
    d = stats.get(fam, [])
    mean = sum(d) / len(d) if d else float("nan")
    print(f"  {fam:14s} launches {len(d):5d}  mean {mean:8.1f} us  per frame {sum(d) / frames:8.1f} us")
