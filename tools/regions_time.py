#!/usr/bin/env python
"""Time quant_recurse of every region of a device-resident tag image, each region to its own palette, with its label
image, three ways in one process:
  host         today's route: pixels and tags to the host, numpy gather by tag (raster order inside a region),
               dq_quant_recurse_batch_ctx, dq_map_colors_batch_ctx with labels, numpy scatter, out and labels back up
  torch        torch gather (stable argsort of the tags), dq_quant_recurse_batch_device, dq_map_colors_batch_device with
               labels, torch scatter: every pixel stays on the device
  regions      one dq_quant_regions_device call with labels (csrc/dq_regions.cu)
  regions_nolab the same without labels
Arms alternate inside every repetition; each is warmed up first and ends in a device synchronisation.  Every arm's
output, palettes, actual K and labels are compared with the host route's.  A separate torch.profiler run of the regions
arm gives the device time of its own kernels (the tag sort, gather, offsets and scatter back) per call.  Prints the card
and its power limit beside the numbers.
Usage: python tools/regions_time.py [reps] [--json FILE]"""
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
OWN_KERNELS = ("region_", "tile_rowscan")


def voronoi(h, w, cells, seed):
    from scipy.spatial import cKDTree
    pts = np.random.default_rng(seed).random((cells, 2)) * [h, w]
    yy, xx = np.mgrid[0:h, 0:w]
    return cKDTree(pts).query(np.c_[yy.ravel(), xx.ravel()])[1].astype(np.uint32)


def workloads(o):
    """(name, pixels, tags, ks)"""
    g1 = o.generate(1, 1920, 1080, 7)
    z = np.load(os.path.join(ROOT, "tests", "golden", "cookie_px.npz"))
    h, w = (int(x) for x in z["shape"][:2])
    cookie = z["px"].ravel().astype(np.uint32)
    yy, xx = np.mgrid[0:h, 0:w]
    tiles = ((yy // 32) * (-(-w // 32)) + xx // 32).ravel().astype(np.uint32)
    cells = voronoi(1080, 1920, 1920 * 1080 // 1000, 1)
    g1_4k = o.generate(1, 3840, 2160, 9)
    scattered = np.random.default_rng(3).integers(0, 2000, g1.size).astype(np.uint32)
    return [
        ("g1_1080p_voronoi1000px_K4", g1, cells, [4] * int(cells.max() + 1)),
        ("g1_1080p_voronoi1000px_K125", g1, cells, [125] * int(cells.max() + 1)),
        ("cookie_32x32_tiles_K16", cookie, tiles, [16] * int(tiles.max() + 1)),
        ("g1_4k_voronoi8000_K4", g1_4k, voronoi(2160, 3840, 8000, 2), [4] * 8000),
        ("g1_1080p_scattered2000_K4", g1, scattered, [4] * 2000),
    ]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def canonical(out, ct, nk, ks, lab):
    """(out, labels, per-region palettes) as numpy, from whichever arm"""
    def host(a):
        return a.cpu().numpy().view(np.uint32) if hasattr(a, "cpu") else np.asarray(a, np.uint32)
    off = np.concatenate([[0], np.cumsum(np.asarray(ks, np.int64))])
    pals = [host(ct)[off[r]:off[r] + int(nk[r])].tobytes() for r in range(len(ks))]
    return host(out), None if lab is None else host(lab), pals


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

    def arm_host(d_px, d_tags, ks):
        px, tags = d_px.cpu().numpy().view(np.uint32), d_tags.cpu().numpy().view(np.uint32)
        num = len(ks)
        inside = tags < num
        counts = np.bincount(tags[inside], minlength=num)
        order = np.argsort(np.where(inside, tags, num), kind="stable")[:int(counts.sum())]
        flat = np.ascontiguousarray(px[order])
        used = counts > 0
        offsets = np.concatenate([[0], np.cumsum(counts[used])]).astype(np.uint32)
        kk = np.asarray(ks, np.uint32)[used].copy()
        ct_items = np.zeros(max(int(kk.astype(np.int64).sum()), 1), np.uint32)
        qout = np.zeros_like(flat)
        req = kk.copy()
        lib.dq_quant_recurse_batch_ctx(ctx, kk.size, pkg._p(offsets), flat.size, pkg._p(flat), pkg._p(qout), pkg._p(kk),
                                       pkg._p(ct_items), 0)
        item_off = np.concatenate([[0], np.cumsum(req.astype(np.int64))])
        packed = np.concatenate([ct_items[item_off[i]:item_off[i] + kk[i]] for i in range(kk.size)])
        mout, mlab = np.zeros_like(flat), np.zeros_like(flat)
        sizes = kk.astype(np.int32)
        lib.dq_map_colors_batch_ctx(ctx, kk.size, pkg._p(offsets), flat.size, pkg._p(flat), pkg._p(mout),
                                    sizes.ctypes.data_as(pkg.C.POINTER(pkg.C.c_int)), pkg._p(packed), pkg._p(mlab))
        out, lab = np.zeros_like(px), np.zeros_like(px)
        out[order], lab[order] = qout, mlab
        # palettes in the regions call's packing (requested K of every region)
        ct = np.zeros(max(int(np.sum(ks)), 1), np.uint32)
        nk = np.zeros(num, np.uint32)
        roff = np.concatenate([[0], np.cumsum(np.asarray(ks, np.int64))])
        for i, r in enumerate(np.flatnonzero(used)):
            ct[roff[r]:roff[r] + kk[i]] = ct_items[item_off[i]:item_off[i] + kk[i]]
            nk[r] = kk[i]
        d_out = torch.from_numpy(out.view(np.int32)).to(dev)
        d_lab = torch.from_numpy(lab.view(np.int32)).to(dev)
        torch.cuda.synchronize()
        return d_out, ct, nk, d_lab

    def arm_torch(d_px, d_tags, ks):
        num = len(ks)
        key = torch.clamp(d_tags.long(), max=num)
        order = torch.argsort(key, stable=True)
        counts = torch.bincount(key, minlength=num + 1)[:num].cpu().numpy()
        m = int(counts.sum())
        order = order[:m]
        flat = d_px[order].contiguous()
        used = counts > 0
        offsets = np.concatenate([[0], np.cumsum(counts[used])]).astype(np.uint32)
        kk = np.asarray(ks, np.uint32)[used]
        qout, ct_items, nk_items = dq.quant_recurse_batch_device(flat, offsets, kk)
        item_off = np.concatenate([[0], np.cumsum(kk.astype(np.int64))])
        pals = [ct_items[item_off[i]:item_off[i] + nk_items[i]] for i in range(kk.size)]
        _, mlab = dq.map_colors_batch_device(flat, offsets, pals, labels=True)
        out, lab = torch.zeros_like(d_px), torch.zeros_like(d_px)
        out[order], lab[order] = qout, mlab
        ct = np.zeros(max(int(np.sum(ks)), 1), np.uint32)
        nk = np.zeros(num, np.uint32)
        roff = np.concatenate([[0], np.cumsum(np.asarray(ks, np.int64))])
        for i, r in enumerate(np.flatnonzero(used)):
            ct[roff[r]:roff[r] + nk_items[i]] = pals[i]
            nk[r] = nk_items[i]
        torch.cuda.synchronize()
        return out, ct, nk, lab

    def arm_regions(d_px, d_tags, ks, labels=True):
        res = dq.quant_regions_device(d_px, d_tags, ks, labels=labels)
        torch.cuda.synchronize()
        return res if labels else (*res, None)

    arms = {"host": arm_host, "torch": arm_torch, "regions": arm_regions,
            "regions_nolab": lambda p, t, k: arm_regions(p, t, k, labels=False)}
    gpu = card()
    print(f"# card: {gpu}")
    results = []
    for name, px, tags, ks in workloads(o):
        d_px = torch.from_numpy(px.view(np.int32)).to(dev)
        d_tags = torch.from_numpy(tags.view(np.int32)).to(dev)
        with muted((2,)):
            ref = None
            for a, fn in arms.items():  # warm-up and equality
                res = fn(d_px, d_tags, ks)
                got = canonical(res[0], res[1], res[2], ks, res[3])
                if ref is None:
                    ref = got
                assert np.array_equal(got[0], ref[0]), f"{name}: {a} output differs from the host route"
                assert got[2] == ref[2], f"{name}: {a} palettes differ from the host route"
                if got[1] is not None:
                    assert np.array_equal(got[1], ref[1]), f"{name}: {a} labels differ from the host route"
            times = {a: [] for a in arms}
            for _ in range(args.reps):
                for a, fn in arms.items():
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    fn(d_px, d_tags, ks)
                    times[a].append((time.perf_counter() - t0) * 1e3)
            st = dq.last_batch_stats()
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    arm_regions(d_px, d_tags, ks)
            own = sum(e.self_device_time_total for e in prof.key_averages() if any(s in e.key for s in OWN_KERNELS)) / 3e3
        row = {"workload": name, "pixels": int(px.size), "regions": len(ks),
               "sort_passes": 1 if len(ks) <= 256 else 2 if len(ks) <= 65536 else 3,
               **{f"{a}_ms": float(np.median(v)) for a, v in times.items()},
               "regions_sort_gather_scatter_ms": own, "batched_items": st["batched_items"],
               "single_call_items": st["single_call_items"], "kernel_launches": st["kernel_launches"]}
        results.append(row)
        print(json.dumps(row))
    if args.json:
        with open(args.json, "w") as f:
            json.dump({"card": gpu, "reps": args.reps, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
