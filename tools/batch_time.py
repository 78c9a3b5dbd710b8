#!/usr/bin/env python
"""Time quant_recurse over many small items three ways, on the same device-resident items in one process:
  loop      one dq_quant_recurse_device call per item
  pipeline  the frame pipeline (12 lanes), one submit_device per item, then flush
  batch     one dq_quant_recurse_batch_device call (csrc/dq_batch.cu)
Arms alternate inside every repetition; each is warmed up first and ends in a device synchronisation.  The outputs of the
three arms are compared item for item.  Prints the card and its power limit beside the numbers, ms per batch, items/s, the
share of the batch call spent in the host's palette handling, and the reference on one core where oracle/_ref is built.
Usage: python tools/batch_time.py [reps] [--json FILE]"""
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
from oracle import Oracle, Reference, muted  # noqa: E402

pkg = importlib.import_module("clusteringsegmentation-1_b200")


def tiles(img, size=32):
    h, w = img.shape
    return [np.ascontiguousarray(img[y:y + size, x:x + size]).ravel() for y in range(0, h, size) for x in range(0, w, size)]


def workloads(o):
    g1 = o.generate(1, 1920, 1080, 7).reshape(1080, 1920)
    z = np.load(os.path.join(ROOT, "tests", "golden", "cookie_px.npz"))
    cookie = z["px"].reshape(tuple(int(x) for x in z["shape"])).astype(np.uint32)
    rng = np.random.default_rng(5)
    flat = g1.ravel()
    ragged, ks = [], []
    for _ in range(1000):  # region-like sizes: mostly small, a long tail
        n = int(min(20000, max(1, rng.lognormal(6.5, 1.0))))
        s = int(rng.integers(0, flat.size - n))
        ragged.append(flat[s:s + n].copy())
        ks.append(int(rng.choice([4, 16, 64, 125])))
    out = []
    for name, img in (("g1_1080p_32x32", g1), ("cookie_32x32", cookie)):
        t = tiles(img)
        for k in (4, 125):
            out.append((f"{name}_K{k}", t, [k] * len(t)))
    out.append(("ragged_1000", ragged, ks))
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
    try:
        ref = Reference()
    except FileNotFoundError:
        ref = None
    ctx = lib.dq_default_context()
    pipe = pkg.FramePipeline(lib, 0, 0, depth=12)
    results = {"card": card(), "reps": args.reps, "workloads": []}
    print("card (name, power limit, max SM clock):", results["card"], flush=True)
    for name, items, ks in workloads(o):
        offsets = np.concatenate([[0], np.cumsum([a.size for a in items])]).astype(np.uint32)
        flat = torch.from_numpy(np.concatenate(items).view(np.int32)).to(dev)
        base = flat.data_ptr()
        outs = {a: torch.empty_like(flat) for a in ("loop", "pipeline", "batch")}
        pal_off = np.concatenate([[0], np.cumsum(ks)]).astype(np.int64)
        pals = {a: np.zeros(int(pal_off[-1]), np.uint32) for a in outs}
        nks = {a: np.zeros(len(items), np.uint32) for a in outs}
        torch.cuda.synchronize()

        def run_loop():
            o_ = outs["loop"].data_ptr()
            ct, nk = pals["loop"], nks["loop"]
            for i, k in enumerate(ks):
                v = C.c_uint32(k)
                lib.dq_quant_recurse_device(ctx, int(offsets[i + 1] - offsets[i]), base + 4 * int(offsets[i]), o_ + 4 * int(offsets[i]),
                                            C.byref(v), pkg._p(ct[pal_off[i]:]), 0)
                nk[i] = v.value

        def run_pipeline():
            o_ = outs["pipeline"].data_ptr()
            ct = pals["pipeline"]
            vs = [C.c_uint32(k) for k in ks]
            views = [ct[pal_off[i]:pal_off[i + 1]] for i in range(len(ks))]
            for i in range(len(ks)):
                pipe.submit_device(base + 4 * int(offsets[i]), o_ + 4 * int(offsets[i]), int(offsets[i + 1] - offsets[i]), views[i], vs[i])
            pipe.flush()
            nks["pipeline"][:] = [v.value for v in vs]

        host_ms = []

        def run_batch():
            nk = np.asarray(ks, np.uint32)
            lib.dq_quant_recurse_batch_device(ctx, len(ks), pkg._p(offsets), int(offsets[-1]), base, outs["batch"].data_ptr(), pkg._p(nk),
                                              pkg._p(pals["batch"]), 0)
            nks["batch"][:] = nk
            host_ms.append(dq.last_batch_stats()["host_palette_ms"])

        arms = {"loop": run_loop, "pipeline": run_pipeline, "batch": run_batch}
        times = {a: [] for a in arms}
        with muted((2,)):
            for f in arms.values():  # warm-up of every shape
                f()
            torch.cuda.synchronize()
            host_ms.clear()
            for r in range(args.reps):
                order = list(arms) if r % 2 == 0 else list(reversed(arms))
                for a in order:
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    arms[a]()
                    torch.cuda.synchronize()
                    times[a].append((time.perf_counter() - t0) * 1e3)
        st = dq.last_batch_stats()
        same = {}
        for a in ("loop", "pipeline"):
            ok = np.array_equal(nks[a], nks["batch"]) and torch.equal(outs[a], outs["batch"])
            ok = ok and all(np.array_equal(pals[a][pal_off[i]:pal_off[i] + nks[a][i]], pals["batch"][pal_off[i]:pal_off[i] + nks["batch"][i]])
                            for i in range(len(ks)))
            same[a] = bool(ok)
        row = {"workload": name, "items": len(items), "pixels": int(offsets[-1]), "batched_items": st["batched_items"],
               "single_call_items": st["single_call_items"], "batch_launches": st["kernel_launches"], "same_outputs": same}
        for a, ts in times.items():
            med = float(np.median(ts))
            row[a] = {"ms_median": round(med, 3), "ms_min": round(float(np.min(ts)), 3), "ms_max": round(float(np.max(ts)), 3),
                      "items_per_s": round(len(items) / med * 1e3, 1)}
        row["batch"]["host_palette_ms_median"] = round(float(np.median(host_ms)), 3)
        row["batch"]["host_palette_share"] = round(float(np.median(host_ms)) / row["batch"]["ms_median"], 3)
        if ref is not None:
            t0 = time.perf_counter()
            with muted():
                for px, k in zip(items, ks):
                    ref.quant_recurse(px, k, 0)
            ms = (time.perf_counter() - t0) * 1e3
            row["reference_1core"] = {"ms": round(ms, 3), "items_per_s": round(len(items) / ms * 1e3, 1)}
        else:
            row["reference_1core"] = "not measured (oracle/_ref not built)"
        results["workloads"].append(row)
        print(json.dumps(row), flush=True)
    pipe.close()
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
