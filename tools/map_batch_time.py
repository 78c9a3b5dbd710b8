#!/usr/bin/env python
"""Time map_colors_mps over many items, each with its own palette, on the same device-resident items in one process:
  loop         one dq_map_colors_device call per item
  batch        one dq_map_colors_batch_device call (csrc/dq_batch.cu)
  loop_labels  the loop plus one dq_colortable_indexes_device call per item (the label image)
  batch_labels one dq_map_colors_batch_device call with labels
Arms alternate inside every repetition; each is warmed up first and ends in a device synchronisation.  The outputs (and
labels) of each loop are compared with its batch item for item.  Prints the card and its power limit beside the numbers,
ms per call, items/s and the share of the batch call spent building the search and label tables on the host.
Usage: python tools/map_batch_time.py [reps] [--json FILE]"""
import argparse
import ctypes as C
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


def tiles(img, size=32):
    h, w = img.shape
    return [np.ascontiguousarray(img[y:y + size, x:x + size]).ravel() for y in range(0, h, size) for x in range(0, w, size)]


def workloads(o, dq):
    """(name, items, palettes).  The palettes of the 1080p tiles come from one quant batch call on those tiles: what a
    caller that quantizes its regions and then maps them gets."""
    g1 = o.generate(1, 1920, 1080, 7).reshape(1080, 1920)
    z = np.load(os.path.join(ROOT, "tests", "golden", "cookie_px.npz"))
    cookie = z["px"].reshape(tuple(int(x) for x in z["shape"])).astype(np.uint32)
    grid = np.load(os.path.join(ROOT, "tests", "golden", "reference_outputs.npz"))["grid125"].astype(np.uint32)
    out = []
    t = tiles(g1)
    for k in (4, 125):
        with muted((2,)):
            pals = [p for _, p in dq.quant_recurse_batch(t, [k] * len(t))]
        out.append((f"g1_1080p_32x32_own_K{k}", t, pals))
    t = tiles(cookie)
    out.append(("cookie_32x32_grid125", t, [grid] * len(t)))
    rng = np.random.default_rng(5)
    flat = g1.ravel()
    ragged, pals = [], []
    for _ in range(1000):  # region-like sizes (tools/batch_time.py): mostly small, a long tail
        n = int(min(20000, max(1, rng.lognormal(6.5, 1.0))))
        s = int(rng.integers(0, flat.size - n))
        ragged.append(flat[s:s + n].copy())
        pals.append(rng.integers(0, 1 << 24, int(rng.choice([4, 16, 64, 125, 256])), dtype=np.uint32))
    out.append(("ragged_1000_random_palettes", ragged, pals))
    frames = [o.generate(1, 1920, 1080, s) for s in (11, 12, 13, 14)]
    out.append(("whole_1080p_x4", frames, [f[rng.integers(0, f.size, k)] for f, k in zip(frames, (16, 64, 125, 256))]))
    return out


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("reps", nargs="?", type=int, default=5)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "needs a GPU: nothing here is measured without one"
    dev = torch.device("cuda:0")
    lib = pkg.load_library()
    lib.dq_set_display_timings(0)
    dq = pkg.DivQuant(lib)
    o = Oracle()
    ctx = lib.dq_default_context()
    results = {"card": card(), "reps": args.reps, "workloads": []}
    print("card (name, power limit, max SM clock):", results["card"], flush=True)
    for name, items, pals in workloads(o, dq):
        offsets = np.concatenate([[0], np.cumsum([a.size for a in items])]).astype(np.uint32)
        sizes = np.asarray([p.size for p in pals], np.int32)
        pal_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        ct = np.ascontiguousarray(np.concatenate(pals), np.uint32)
        flat = torch.from_numpy(np.concatenate(items).view(np.int32)).to(dev)
        base = flat.data_ptr()
        arms_ = ("loop", "batch", "loop_labels", "batch_labels")
        outs = {a: torch.empty_like(flat) for a in arms_}
        labs = {a: torch.empty_like(flat) for a in ("loop_labels", "batch_labels")}
        torch.cuda.synchronize()
        cts = [pkg._p(ct[pal_off[i]:]) for i in range(len(items))]
        sizes_p = sizes.ctypes.data_as(C.POINTER(C.c_int))

        def loop(a, labels):
            o_ = outs[a].data_ptr()
            l_ = labs[a].data_ptr() if labels else 0
            for i in range(len(items)):
                b, n = 4 * int(offsets[i]), int(offsets[i + 1] - offsets[i])
                lib.dq_map_colors_device(ctx, base + b, n, o_ + b, cts[i], int(sizes[i]), 1)
                if labels:
                    lib.dq_colortable_indexes_device(ctx, o_ + b, n, cts[i], int(sizes[i]), l_ + b, 0)

        host_ms = {"batch": [], "batch_labels": []}

        def batch(a, labels):
            lib.dq_map_colors_batch_device(ctx, len(items), pkg._p(offsets), int(offsets[-1]), base, outs[a].data_ptr(), sizes_p,
                                           pkg._p(ct), labs[a].data_ptr() if labels else None)
            host_ms[a].append(dq.last_batch_stats()["host_palette_ms"])

        arms = {"loop": lambda: loop("loop", False), "batch": lambda: batch("batch", False),
                "loop_labels": lambda: loop("loop_labels", True), "batch_labels": lambda: batch("batch_labels", True)}
        times = {a: [] for a in arms}
        for f in arms.values():  # warm-up of every shape
            f()
        torch.cuda.synchronize()
        for v in host_ms.values():
            v.clear()
        stats = {}
        for r in range(args.reps):
            order = list(arms) if r % 2 == 0 else list(reversed(arms))
            for a in order:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                arms[a]()
                torch.cuda.synchronize()
                times[a].append((time.perf_counter() - t0) * 1e3)
                if a.startswith("batch"):
                    stats[a] = dq.last_batch_stats()
        same = {"outputs": bool(torch.equal(outs["loop"], outs["batch"])),
                "outputs_with_labels": bool(torch.equal(outs["loop_labels"], outs["batch_labels"])),
                "labels": bool(torch.equal(labs["loop_labels"], labs["batch_labels"])),
                "outputs_labels_vs_plain": bool(torch.equal(outs["batch"], outs["batch_labels"]))}
        st = stats["batch"]
        row = {"workload": name, "items": len(items), "pixels": int(offsets[-1]), "batched_items": st["batched_items"],
               "single_call_items": st["single_call_items"], "batch_launches": st["kernel_launches"],
               "batch_labels_launches": stats["batch_labels"]["kernel_launches"], "same": same}
        for a, ts in times.items():
            med = float(np.median(ts))
            row[a] = {"ms_median": round(med, 3), "ms_min": round(float(np.min(ts)), 3), "ms_max": round(float(np.max(ts)), 3),
                      "items_per_s": round(len(items) / med * 1e3, 1)}
        for a, v in host_ms.items():
            row[a]["host_palette_ms_median"] = round(float(np.median(v)), 3)
            row[a]["host_palette_share"] = round(float(np.median(v)) / row[a]["ms_median"], 3)
        results["workloads"].append(row)
        print(json.dumps(row), flush=True)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(results, f, indent=1)
    if not all(all(r["same"].values()) for r in results["workloads"]):
        sys.exit("arms disagree")


if __name__ == "__main__":
    main()
