#!/usr/bin/env python
"""Row-sharded quant_recurse of one image over the ranks of a torchrun job (dq_rows_*: one grouped ncclAllGather per
image inside the library, no host wait before the palette), checked against the single-GPU result of the whole image and
timed next to it.
With a seed, the image is G1 of that seed; where tests/golden/frames.npz holds the compiled reference's fingerprint of that
image (1920x1080 K=64, 3840x2160 K=256), the single-GPU result is checked against it as well.
usage: torchrun --nproc-per-node N tools/rows_check.py [w h K reps [seed]]"""
import ctypes as C
import importlib
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import Oracle  # generator only

w, h, k, reps, seed = [int(x) for x in (sys.argv[1:6] + ["3840", "2160", "256", "10", "12345"][len(sys.argv) - 1:])]
rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
pkg = importlib.import_module("clusteringsegmentation-1_b200")
lib = pkg.load_library()
lib.dq_set_display_timings(0)
ctx = lib.dq_context_create(local)
oracle = Oracle()
img = oracle.generate(1, w, h, seed)
r0, r1 = pkg.rows_for_rank(h, world, rank)
shard = torch.from_numpy(img[r0 * w:r1 * w].view(np.int32).copy()).cuda()
d = dist if world > 1 else None
rows = pkg.RowShards(lib, ctx, d, list_capacity=1 << 18)
out, pal = rows.quant_recurse(shard, w * h, k)
# reference: the whole image on this GPU alone
full = torch.from_numpy(img.view(np.int32)).cuda()
full_out = torch.empty_like(full)
ct = np.zeros(k, np.uint32)
nk = C.c_uint32(k)
u32p = C.POINTER(C.c_uint32)


def single():
    nk.value = k
    lib.dq_quant_recurse_device(ctx, full.numel(), full.data_ptr(), full_out.data_ptr(), C.byref(nk), ct.ctypes.data_as(u32p), 0)


single()
ok = np.array_equal(pal, ct[:nk.value]) and torch.equal(out, full_out[r0 * w:r1 * w])
golden = None
tag = {(1920, 1080, 64): "c4", (3840, 2160, 256): "bench"}.get((w, h, k))
if tag:
    frames = np.load(os.path.join(ROOT, "tests", "golden", "frames.npz"))
    at = np.nonzero(frames[f"{tag}_seeds"] == seed)[0]
    if at.size:
        i = int(at[0])
        golden = (ct[:nk.value].size == int(frames[f"{tag}_pal_size"][i]) and
                  oracle.hash_words(ct[:nk.value]) == int(frames[f"{tag}_pal_hash"][i]) and
                  oracle.hash_words(full_out.cpu().numpy().view(np.uint32)) == int(frames[f"{tag}_out_hash"][i]))


def timed(fn):
    """max over ranks of the device time per call (CUDA events on torch's stream bracket the library's stream: the
    library's calls are synchronous with respect to the host)."""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    if d:
        d.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / reps], device="cuda")
    if d:
        d.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


ms_lib = timed(lambda: rows.quant_recurse(shard, w * h, k, out))
ms_one = timed(single)
flag = torch.tensor([1 if ok else 0], device="cuda")
if d:
    d.all_reduce(flag, op=dist.ReduceOp.MIN)
if rank == 0:
    verdict = "bit-exact vs single GPU" if flag.item() else "MISMATCH"
    verdict += {None: "", True: ", reference fingerprint ok", False: ", reference fingerprint MISMATCH"}[golden]
    print(f"rows x{world} {w}x{h} K={k} seed {seed}: {verdict}; {ms_lib:.3f} ms/image, one GPU alone {ms_one:.3f}",
          flush=True)
rows.close()
if d:
    d.destroy_process_group()
sys.exit(0 if flag.item() and golden is not False else 1)
