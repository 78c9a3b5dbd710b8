#!/usr/bin/env python
"""Time map_colors_mps of every region of a device-resident tag image, each region to its own palette, with its label
image, four ways in one process:
  host          the route without the call: pixels and tags to the host, numpy gather by tag (raster order inside a
                region), dq_map_colors_batch_ctx with labels, numpy scatter, out and labels back up
  torch         torch gather (stable argsort of the tags), dq_map_colors_batch_device with labels, torch scatter: every
                pixel stays on the device
  regions       one dq_map_regions_device call with labels (csrc/dq_regions.cu, then the batch remap)
  regions_nolab the same without labels
The palettes are made as the reference's region loop makes them: each region's palette from dq_quant_regions, then
reversed with one entry dropped (the re-sorted and edited palettes of ClusteringSegmentation.cpp:3816 / :2434), or the
fixed grid-125 palette for every tile.  Arms alternate inside every repetition; each is warmed up first and ends in a
device synchronisation.  Every arm's output and labels are compared with the host route's before timing.  A separate
torch.profiler run of the regions arm gives the device time of the partition kernels (tag sort, gather, offsets, scatter
back) and of the batch remap per call.  Prints the card and its power limit beside the numbers.
Usage: python tools/map_regions_time.py [reps] [--json FILE]"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import Oracle, muted  # noqa: E402

pkg = importlib.import_module("clusteringsegmentation-1_b200")
PARTITION_KERNELS = ("region_", "tile_rowscan")
REMAP_KERNELS = ("batch_remap",)


def voronoi(h, w, cells, seed):
    from scipy.spatial import cKDTree
    pts = np.random.default_rng(seed).random((cells, 2)) * [h, w]
    yy, xx = np.mgrid[0:h, 0:w]
    return cKDTree(pts).query(np.c_[yy.ravel(), xx.ravel()])[1].astype(np.uint32)


def edited_palettes(dq, px, tags, num, k):
    """Each region's palette from dq_quant_regions, reversed with one entry dropped (empty for a region without pixels)."""
    with muted((2,)):
        _, ct, nk = dq.quant_regions(px, tags, [k] * num)
    off = np.concatenate([[0], np.cumsum(np.full(num, k, np.int64))])
    return [ct[off[r]:off[r] + nk[r]][::-1][:max(int(nk[r]) - 1, 1) if nk[r] else 0].copy() for r in range(num)]


def workloads(dq, o):
    """(name, pixels, tags, palettes)"""
    g1 = o.generate(1, 1920, 1080, 7)
    z = np.load(os.path.join(ROOT, "tests", "golden", "cookie_px.npz"))
    h, w = (int(x) for x in z["shape"][:2])
    cookie = z["px"].ravel().astype(np.uint32)
    yy, xx = np.mgrid[0:h, 0:w]
    tiles = ((yy // 32) * (-(-w // 32)) + xx // 32).ravel().astype(np.uint32)
    grid = np.load(os.path.join(ROOT, "tests", "golden", "reference_outputs.npz"))["grid125"].astype(np.uint32)
    cells = voronoi(1080, 1920, 1920 * 1080 // 1000, 1)
    g1_4k = o.generate(1, 3840, 2160, 9)
    cells_4k = voronoi(2160, 3840, 8000, 2)
    scattered = np.random.default_rng(3).integers(0, 2000, g1.size).astype(np.uint32)
    nc = int(cells.max() + 1)
    return [
        ("g1_1080p_voronoi1000px_K4_edited", g1, cells, edited_palettes(dq, g1, cells, nc, 4)),
        ("g1_1080p_voronoi1000px_K125_edited", g1, cells, edited_palettes(dq, g1, cells, nc, 125)),
        ("cookie_32x32_tiles_grid125", cookie, tiles, [grid] * int(tiles.max() + 1)),
        ("g1_4k_voronoi8000_K4_edited", g1_4k, cells_4k, edited_palettes(dq, g1_4k, cells_4k, 8000, 4)),
        ("g1_1080p_scattered2000_K4_edited", g1, scattered, edited_palettes(dq, g1, scattered, 2000, 4)),
    ]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def host_np(a):
    return a.cpu().numpy().view(np.uint32) if hasattr(a, "cpu") else np.asarray(a, np.uint32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("reps", nargs="?", type=int, default=5)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "needs a GPU: nothing here is measured without one"
    dev = torch.device("cuda:0")
    dq = pkg.DivQuant(timings=False)
    lib, ctx = dq.lib, dq.lib.dq_default_context()
    o = Oracle()

    def items_of(counts, pals):
        """the mapped regions with pixels: (mask over regions, offsets, sizes, packed palettes)"""
        used = (counts > 0) & np.array([p.size > 0 for p in pals])
        offsets = np.concatenate([[0], np.cumsum(counts[used])]).astype(np.uint32)
        sel = [pals[r] for r in np.flatnonzero(used)]
        sizes = np.asarray([p.size for p in sel], np.int32)
        return used, offsets, sizes, np.concatenate(sel + [np.zeros(1, np.uint32)])

    def arm_host(d_px, d_tags, pals):
        px, tags = d_px.cpu().numpy().view(np.uint32), d_tags.cpu().numpy().view(np.uint32)
        num = len(pals)
        inside = tags < num
        counts = np.bincount(tags[inside], minlength=num)
        order = np.argsort(np.where(inside, tags, num), kind="stable")[:int(counts.sum())]
        used, offsets, sizes, ct = items_of(counts, pals)
        keep = np.repeat(used, counts)  # drop the pixels of unmapped regions
        order = order[keep]
        flat = np.ascontiguousarray(px[order])
        mout, mlab = np.zeros_like(flat), np.zeros_like(flat)
        lib.dq_map_colors_batch_ctx(ctx, sizes.size, pkg._p(offsets), flat.size, pkg._p(flat), pkg._p(mout),
                                    sizes.ctypes.data_as(pkg.C.POINTER(pkg.C.c_int)), pkg._p(ct), pkg._p(mlab))
        out, lab = np.zeros_like(px), np.zeros_like(px)
        out[order], lab[order] = mout, mlab
        d_out = torch.from_numpy(out.view(np.int32)).to(dev)
        d_lab = torch.from_numpy(lab.view(np.int32)).to(dev)
        torch.cuda.synchronize()
        return d_out, d_lab

    def arm_torch(d_px, d_tags, pals):
        num = len(pals)
        key = torch.clamp(d_tags.long(), max=num)
        order = torch.argsort(key, stable=True)
        counts = torch.bincount(key, minlength=num + 1)[:num].cpu().numpy()
        order = order[:int(counts.sum())]
        used, offsets, sizes, ct = items_of(counts, pals)
        if not used.all():
            order = order[torch.from_numpy(np.repeat(used, counts)).to(dev)]
        flat = d_px[order].contiguous()
        mout, mlab = torch.empty_like(flat), torch.empty_like(flat)
        torch.cuda.current_stream(dev).synchronize()
        lib.dq_map_colors_batch_device(ctx, sizes.size, pkg._p(offsets), flat.numel(), flat.data_ptr(), mout.data_ptr(),
                                       sizes.ctypes.data_as(pkg.C.POINTER(pkg.C.c_int)), pkg._p(ct), mlab.data_ptr())
        out, lab = torch.zeros_like(d_px), torch.zeros_like(d_px)
        out[order], lab[order] = mout, mlab
        torch.cuda.synchronize()
        return out, lab

    def arm_regions(d_px, d_tags, pals, labels=True):
        res = dq.map_regions_device(d_px, d_tags, pals, labels=labels)
        torch.cuda.synchronize()
        return res if labels else (res, None)

    arms = {"host": arm_host, "torch": arm_torch, "regions": arm_regions,
            "regions_nolab": lambda p, t, k: arm_regions(p, t, k, labels=False)}
    gpu = card()
    print(f"# card: {gpu}")
    results = []
    for name, px, tags, pals in workloads(dq, o):
        d_px = torch.from_numpy(px.view(np.int32)).to(dev)
        d_tags = torch.from_numpy(tags.view(np.int32)).to(dev)
        ref = None
        for a, fn in arms.items():  # warm-up and equality
            out, lab = fn(d_px, d_tags, pals)
            out, lab = host_np(out), None if lab is None else host_np(lab)
            if ref is None:
                ref = (out, lab)
            assert np.array_equal(out, ref[0]), f"{name}: {a} output differs from the host route"
            if lab is not None:
                assert np.array_equal(lab, ref[1]), f"{name}: {a} labels differ from the host route"
        times = {a: [] for a in arms}
        for _ in range(args.reps):
            for a, fn in arms.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn(d_px, d_tags, pals)
                times[a].append((time.perf_counter() - t0) * 1e3)
        arm_regions(d_px, d_tags, pals)
        st = dq.last_batch_stats()
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                arm_regions(d_px, d_tags, pals)

        def device_ms(keys):
            return sum(e.self_device_time_total for e in prof.key_averages() if any(s in e.key for s in keys)) / 3e3
        row = {"workload": name, "pixels": int(px.size), "regions": len(pals),
               "sort_passes": 1 if len(pals) <= 256 else 2 if len(pals) <= 65536 else 3,
               "palette_entries": int(sum(p.size for p in pals)),
               **{f"{a}_ms": float(np.median(v)) for a, v in times.items()},
               "regions_partition_scatter_ms": device_ms(PARTITION_KERNELS), "regions_batch_remap_ms": device_ms(REMAP_KERNELS),
               "host_palette_ms": st["host_palette_ms"], "batched_items": st["batched_items"],
               "single_call_items": st["single_call_items"], "kernel_launches": st["kernel_launches"]}
        results.append(row)
        print(json.dumps(row))
    if args.json:
        with open(args.json, "w") as f:
            json.dump({"card": gpu, "reps": args.reps, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
