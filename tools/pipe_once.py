#!/usr/bin/env python
"""A few frames through the frame pipeline (for ncu launch lists of its kernels).
usage: python tools/pipe_once.py [width height K frames lanes]"""
import ctypes as C
import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import Oracle  # input generator only

w, h, k, frames, lanes = [int(x) for x in (sys.argv[1:6] + ["3840", "2160", "256", "4", "1"][len(sys.argv) - 1:])]
pkg = importlib.import_module("clusteringsegmentation-1_b200")
lib = pkg.load_library()
lib.dq_set_display_timings(0)
n = w * h
o = Oracle()
dev = [torch.from_numpy(o.generate(1, w, h, 12345 + s).view(np.int32)).cuda() for s in range(min(frames, 6))]
outs = [torch.empty(n, dtype=torch.int32, device="cuda") for _ in range(frames)]
pipe = lib.dq_pipeline_create_lanes(0, 0, lanes, 0)
u32p = C.POINTER(C.c_uint32)
nks = [C.c_uint32(k) for _ in range(frames)]
cts = [np.zeros(k, np.uint32) for _ in range(frames)]
for i in range(frames):
    lib.dq_pipeline_submit_device(pipe, n, dev[i % len(dev)].data_ptr(), outs[i].data_ptr(), C.byref(nks[i]), cts[i].ctypes.data_as(u32p), 0)
lib.dq_pipeline_flush(pipe)
print("ms/frame", lib.dq_pipeline_last_elapsed_ms(pipe) / frames, "k", [x.value for x in nks], "flagged", lib.dq_pipeline_flagged_frames(pipe))
lib.dq_pipeline_destroy(pipe)
