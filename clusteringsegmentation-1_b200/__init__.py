"""clusteringsegmentation-1_b200 -- B200-native DivQuant colour quantizer (host-side Python mirror).

The product is ``libdivquant_b200.so`` (hand-written CUDA for sm_100a behind the C ABI declared in
``include/divquant_b200.h``).  This module is a thin ctypes mirror of the reference's interface for
that path (``quant_recurse``, ``quant_varpart_fast``, ``map_colors_mps``, ``calc_color_table``,
``cut_bits`` -- DivQuant/DivQuantHeader.h:52-96, DivQuant/quant_util.h:10) used by ``tests/`` and
``bench.py``.  It never computes anything itself and has no CPU fallback: if the shared library is
missing it raises, and the library aborts when there is no sm_100a device.

The directory name is not a Python identifier; import it with
``importlib.import_module("clusteringsegmentation-1_b200")``.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdivquant_b200.so")
INCLUDE_DIR = os.path.join(os.path.dirname(_HERE), "include")

_u32p = C.POINTER(C.c_uint32)
_f64p = C.POINTER(C.c_double)


class SplitRecord(C.Structure):
    """dq_split_record (include/divquant_b200.h), same fields as the oracle's record."""
    _fields_ = [("new_index", C.c_int32), ("old_index", C.c_int32), ("cut_axis", C.c_int32),
                ("num_points", C.c_int32), ("new_size", C.c_int32), ("is_last", C.c_int32),
                ("cut_pos", C.c_double), ("total_weight", C.c_double), ("new_weight", C.c_double),
                ("old_weight", C.c_double), ("new_mean", C.c_double * 3), ("old_mean", C.c_double * 3),
                ("new_var", C.c_double * 3), ("old_var", C.c_double * 3), ("new_tse", C.c_double),
                ("old_tse", C.c_double)]


class CallStats(C.Structure):
    _fields_ = [("num_pixels", C.c_uint32), ("num_points", C.c_uint32), ("requested_colors", C.c_uint32),
                ("actual_colors", C.c_uint32), ("empty_clusters", C.c_uint32), ("split_rounds", C.c_uint32),
                ("splits_computed", C.c_uint32), ("remap_path", C.c_uint32), ("kernel_launches", C.c_uint32),
                ("stage_ms", C.c_float * 7), ("tie_flags", C.c_uint32), ("ordered_rerun", C.c_uint32),
                ("tie_resolved", C.c_uint32), ("cut_overrides", C.c_uint32)]

    STAGES = ("hist_insert", "hist_collect", "split", "map_unique_or_bruteforce", "map_gather", "table_clear", "total")

    def as_dict(self):
        d = {n: getattr(self, n) for n, _ in self._fields_ if n != "stage_ms"}
        d["stage_ms"] = {s: float(self.stage_ms[i]) for i, s in enumerate(self.STAGES)}
        return d


class BatchStats(C.Structure):
    """dq_batch_stats: which path the items of the last batch call took."""
    _fields_ = [("items", C.c_uint32), ("batched_items", C.c_uint32), ("single_call_items", C.c_uint32),
                ("empty_clusters", C.c_uint32), ("kernel_launches", C.c_uint32), ("host_palette_ms", C.c_float)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


def build(verbose=False):
    """Compile libdivquant_b200.so in-tree (nvcc, sm_100a only)."""
    subprocess.run(["make", "-C", _HERE, "-j4"], check=True, stdout=None if verbose else subprocess.DEVNULL)


def load_library(path=LIB_PATH):
    path = os.environ.get("DIVQUANT_B200_LIB", path)  # (A/B timing of two builds on one box: tools/)
    if not os.path.exists(path):
        raise FileNotFoundError(
            f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (there is no CPU fallback)")
    lib = C.CDLL(path)
    vp = C.c_void_p
    sigs = {
        "dq_version": (C.c_char_p, []),
        "dq_quant_recurse": (None, [C.c_uint32, _u32p, _u32p, _u32p, _u32p, C.c_int]),
        "dq_quant_varpart_fast": (None, [C.c_uint32, _u32p, _u32p, C.c_uint32, C.c_uint32, _u32p, _u32p, C.c_int,
                                         C.c_int, C.c_int, C.c_int]),
        "dq_map_colors_mps": (None, [_u32p, C.c_uint32, _u32p, _u32p, C.c_int]),
        "dq_calc_color_table": (C.c_int, [_u32p, C.c_uint32, _u32p, C.c_uint32, C.c_uint32, C.c_int,
                                          C.POINTER(C.c_int), _f64p]),
        "dq_cut_bits": (None, [_u32p, C.c_uint32, _u32p, C.c_ubyte, C.c_ubyte, C.c_ubyte]),
        "dq_get_double_scale": (C.c_double, [_u32p, C.c_uint32]),
        "dq_validate_num_bits": (C.c_int, [C.c_ubyte]),
        "dq_set_display_timings": (None, [C.c_int]),
        "dq_context_create": (vp, [C.c_int]),
        "dq_context_destroy": (None, [vp]),
        "dq_default_context": (vp, []),
        "dq_context_stream": (vp, [vp]),
        "dq_context_synchronize": (None, [vp]),
        "dq_context_last_stats": (None, [vp, C.POINTER(CallStats)]),
        "dq_context_set_profiling": (None, [vp, C.c_int]),
        "dq_quant_recurse_device": (None, [vp, C.c_uint32, vp, vp, _u32p, _u32p, C.c_int]),
        "dq_map_colors_device": (None, [vp, vp, C.c_uint32, vp, _u32p, C.c_int, C.c_int]),
        "dq_quant_varpart_device": (None, [vp, C.c_uint32, vp, C.c_uint32, C.c_uint32, _u32p, _u32p, C.c_int,
                                           C.c_int, C.c_int, C.c_int]),
        "dq_quant_recurse_ctx": (None, [vp, C.c_uint32, _u32p, _u32p, _u32p, _u32p, C.c_int]),
        "dq_quant_recurse_batch_device": (None, [vp, C.c_uint32, _u32p, C.c_uint32, vp, vp, _u32p, _u32p, C.c_int]),
        "dq_quant_recurse_batch_ctx": (None, [vp, C.c_uint32, _u32p, C.c_uint32, _u32p, _u32p, _u32p, _u32p, C.c_int]),
        "dq_context_last_batch_stats": (None, [vp, C.POINTER(BatchStats)]),
        "dq_map_colors_batch_device": (None, [vp, C.c_uint32, _u32p, C.c_uint32, vp, vp, C.POINTER(C.c_int), _u32p, vp]),
        "dq_map_colors_batch_ctx": (None, [vp, C.c_uint32, _u32p, C.c_uint32, _u32p, _u32p, C.POINTER(C.c_int), _u32p, _u32p]),
        "dq_quant_regions_device": (None, [vp, C.c_uint32, vp, vp, C.c_uint32, vp, _u32p, _u32p, vp]),
        "dq_quant_regions_ctx": (None, [vp, C.c_uint32, _u32p, _u32p, C.c_uint32, _u32p, _u32p, _u32p, _u32p]),
        "dq_map_regions_device": (None, [vp, C.c_uint32, vp, vp, C.c_uint32, C.POINTER(C.c_int), _u32p, vp, vp]),
        "dq_map_regions_ctx": (None, [vp, C.c_uint32, _u32p, _u32p, C.c_uint32, C.POINTER(C.c_int), _u32p, _u32p, _u32p]),
        "dq_context_set_split_ctas": (None, [vp, C.c_int]),
        "dq_context_set_exact_small": (None, [vp, C.c_int]),
        "dq_context_set_exact_max_points": (None, [vp, C.c_uint32]),
        "dq_context_set_tie_policy": (None, [vp, C.c_int]),
        "dq_srm_num_pairs": (C.c_uint32, [C.c_uint32, C.c_uint32]),
        "dq_srm_sorted_edges": (None, [vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, vp]),
        "dq_srm_sorted_edges_device": (None, [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, vp]),
        "dq_pixel_histogram": (C.c_uint32, [_u32p, C.c_uint32, _u32p, _u32p, C.c_uint32]),
        "dq_block_vote": (None, [_u32p, C.c_uint32, C.c_uint32, C.c_uint32, _u32p]),
        "dq_block_vote_device": (None, [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, vp]),
        "dq_quant_blocks": (None, [_u32p, C.c_uint32, C.c_uint32, C.c_uint32, _u32p, C.c_int, _u32p, _u32p]),
        "dq_colortable_indexes": (None, [_u32p, C.c_uint32, _u32p, C.c_int, _u32p, C.c_int]),
        "dq_colortable_indexes_device": (None, [vp, vp, C.c_uint32, _u32p, C.c_int, vp, C.c_int]),
        "dq_rows_unique_id": (None, [vp]),
        "dq_rows_create": (vp, [vp, C.c_int, C.c_int, vp, C.c_uint32]),
        "dq_rows_destroy": (None, [vp]),
        "dq_rows_quant_recurse": (None, [vp, vp, C.c_uint32, C.c_uint64, vp, _u32p, _u32p]),
        "dq_pipeline_create": (vp, [C.c_int, C.c_uint32, C.c_int]),
        "dq_pipeline_destroy": (None, [vp]),
        "dq_pipeline_create_lanes": (vp, [C.c_int, C.c_uint32, C.c_int, C.c_int]),
        "dq_pipeline_submit": (C.c_uint64, [vp, C.c_uint32, _u32p, _u32p, _u32p, _u32p, C.c_int]),
        "dq_pipeline_submit_device": (C.c_uint64, [vp, C.c_uint32, vp, vp, _u32p, _u32p, C.c_int]),
        "dq_pipeline_wait": (None, [vp, C.c_uint64]),
        "dq_pipeline_lanes": (C.c_int, [vp]),
        "dq_pipeline_set_blocking_wait": (None, [vp, C.c_int]),
        "dq_pipeline_flush": (None, [vp]),
        "dq_pipeline_last_elapsed_ms": (C.c_float, [vp]),
        "dq_pipeline_context": (vp, [vp]),
        "dq_pipeline_kernel_launches": (C.c_uint64, [vp]),
        "dq_pipeline_flagged_frames": (C.c_uint64, [vp]),
        "dq_pipeline_resolved_frames": (C.c_uint64, [vp]),
        "dq_pipeline_rerun_frames": (C.c_uint64, [vp]),
        "dq_debug_split_points": (C.c_uint32, [vp, _u32p, _u32p, C.c_uint32, C.c_double, C.c_uint32, C.c_int, C.c_int,
                                               _u32p, C.POINTER(SplitRecord), _f64p, _u32p]),
        "dq_debug_histogram": (C.c_uint32, [vp, _u32p, C.c_uint32, _u32p, _u32p]),
        "dq_debug_split_timeline": (C.c_uint32, [vp, C.c_int, C.POINTER(C.c_uint64), C.c_uint32]),
        "dq_host_dedup_palette": (C.c_uint32, [_u32p, C.c_uint32]),
        "dq_host_select_cut_overrides": (C.c_uint32, [_u32p, _u32p, _u32p, C.c_uint32, C.c_uint32, _u32p]),
        "dq_host_build_search_tables": (None, [_u32p, C.c_int, _u32p, C.POINTER(C.c_int32)]),
        "dq_host_build_label_table": (None, [_u32p, C.c_int, _u32p]),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


EXPORTED_C_SYMBOLS = [
    "dq_version", "dq_quant_recurse", "dq_quant_varpart_fast", "dq_map_colors_mps", "dq_calc_color_table", "dq_cut_bits",
    "dq_get_double_scale", "dq_validate_num_bits", "dq_set_display_timings", "dq_context_create", "dq_context_destroy",
    "dq_default_context", "dq_context_stream", "dq_context_synchronize", "dq_context_last_stats", "dq_context_set_profiling",
    "dq_quant_recurse_device", "dq_map_colors_device", "dq_quant_varpart_device", "dq_quant_recurse_ctx",
    "dq_srm_num_pairs", "dq_srm_sorted_edges", "dq_srm_sorted_edges_device", "dq_context_set_split_ctas", "dq_context_set_exact_small", "dq_context_set_exact_max_points", "dq_context_set_tie_policy", "dq_pixel_histogram", "dq_block_vote", "dq_block_vote_device", "dq_quant_blocks", "dq_colortable_indexes", "dq_colortable_indexes_device", "dq_rows_unique_id", "dq_rows_create", "dq_rows_destroy", "dq_rows_quant_recurse", "dq_pipeline_create", "dq_pipeline_create_lanes", "dq_pipeline_destroy", "dq_pipeline_submit", "dq_pipeline_submit_device", "dq_pipeline_wait", "dq_pipeline_lanes", "dq_pipeline_set_blocking_wait", "dq_pipeline_flush", "dq_pipeline_last_elapsed_ms",
    "dq_pipeline_context", "dq_pipeline_kernel_launches", "dq_pipeline_flagged_frames",
    "dq_pipeline_resolved_frames", "dq_pipeline_rerun_frames",
    "dq_quant_recurse_batch_device", "dq_quant_recurse_batch_ctx", "dq_context_last_batch_stats",
    "dq_map_colors_batch_device", "dq_map_colors_batch_ctx", "dq_quant_regions_device", "dq_quant_regions_ctx",
    "dq_map_regions_device", "dq_map_regions_ctx",
    "dq_debug_split_points", "dq_debug_histogram", "dq_debug_split_timeline", "dq_host_dedup_palette", "dq_host_build_search_tables", "dq_host_select_cut_overrides",
    "dq_host_build_label_table",
]

# The reference's own symbol names (SURVEY.md 8b), exported for relinking the reference's callers.
REFERENCE_SYMBOLS = [
    "_Z18quant_varpart_fastjPKjPjjjS1_S1_iiii", "_Z14map_colors_mpsPKjjPjS1_i", "_Z16calc_color_tablePKjjPjjjiPi",
    "_Z16get_double_scalePKjj", "_Z8cut_bitsPKjjPjhhh", "_Z17validate_num_bitsh", "_Z9check_memi", "_Z11start_timerv",
    "_Z10stop_timerl", "_Z8timediffll", "quant_recurse",
]


def _u32(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.uint32).ravel())


def _p(a, t=_u32p):
    return a.ctypes.data_as(t)


class DivQuant:
    """Host-pointer mirror of the reference entry points (numpy in, numpy out)."""

    def __init__(self, lib=None, timings=False):
        self.lib = lib or load_library()
        self.lib.dq_set_display_timings(1 if timings else 0)

    # -- reference entry points ----------------------------------------------------------------
    def quant_recurse(self, pixels, k, all_unique=0):
        px = _u32(pixels)
        out = np.zeros_like(px)
        ct = np.zeros(max(int(k), 1), np.uint32)
        nk = C.c_uint32(k)
        self.lib.dq_quant_recurse(px.size, _p(px), _p(out), C.byref(nk), _p(ct), all_unique)
        return out, ct[:nk.value].copy()

    def quant_varpart_fast(self, pixels, k, num_bits=8, dec_factor=1, max_iters=10, all_unique=0, rows=1, cols=None):
        px = _u32(pixels)
        cols = px.size if cols is None else cols
        tmp = np.zeros_like(px)
        ct = np.zeros(max(int(k), 1), np.uint32)
        nk = C.c_uint32(k)
        self.lib.dq_quant_varpart_fast(px.size, _p(px), _p(tmp), rows, cols, C.byref(nk), _p(ct), num_bits, dec_factor,
                                       max_iters, all_unique)
        return ct[:nk.value].copy(), int(k) - nk.value

    def quant_recurse_batch(self, items, ks, all_unique=0, ctx=None):
        """quant_recurse of every pixel set in `items` (uint32 arrays) with the K in `ks`, in one call
        (dq_quant_recurse_batch_ctx).  Returns a list of (out, palette), one per item, each equal to
        quant_recurse(items[i], ks[i], all_unique) on the same context."""
        arrs = [_u32(a) for a in items]
        ks = [int(k) for k in ks]
        if len(arrs) != len(ks):
            raise ValueError("one K per item")
        if not arrs:
            return []
        offsets = np.zeros(len(arrs) + 1, np.uint32)
        np.cumsum([a.size for a in arrs], out=offsets[1:])
        flat = np.concatenate(arrs) if offsets[-1] else np.zeros(1, np.uint32)
        out = np.zeros_like(flat)
        nk = np.asarray(ks, np.uint32)
        pal_off = np.concatenate([[0], np.cumsum(ks)]).astype(np.int64)
        ct = np.zeros(max(int(pal_off[-1]), 1), np.uint32)
        self.lib.dq_quant_recurse_batch_ctx(ctx or self.lib.dq_default_context(), len(arrs), _p(offsets), flat.size, _p(flat), _p(out),
                                            _p(nk), _p(ct), all_unique)
        return [(out[offsets[i]:offsets[i + 1]].copy(), ct[pal_off[i]:pal_off[i] + nk[i]].copy()) for i in range(len(arrs))]

    def quant_recurse_batch_device(self, flat, offsets, ks, all_unique=0, ctx=None, out=None):
        """Device form (dq_quant_recurse_batch_device): `flat` is a CUDA tensor of 32-bit pixels holding the items end to
        end, item i = flat[offsets[i]:offsets[i+1]].  Returns (out tensor, palettes, actual K): palettes is the uint32
        array of sum(ks) words in which item i's palette starts at sum(ks[:i]) and holds actual_k[i] entries."""
        import torch
        offs = _u32(offsets)
        nk = _u32(ks).copy()
        if offs.size != nk.size + 1:
            raise ValueError("offsets need one entry more than ks")
        if flat.dtype not in (torch.int32, torch.uint32) or not flat.is_cuda or not flat.is_contiguous():
            raise ValueError("flat must be a contiguous CUDA tensor of 32-bit pixels")
        out = torch.empty_like(flat) if out is None else out
        ct = np.zeros(max(int(nk.astype(np.int64).sum()), 1), np.uint32)
        if nk.size:
            torch.cuda.current_stream(flat.device).synchronize()  # the library works on its context's stream
            self.lib.dq_quant_recurse_batch_device(ctx or self.lib.dq_default_context(), nk.size, _p(offs), flat.numel(),
                                                   flat.data_ptr(), out.data_ptr(), _p(nk), _p(ct), all_unique)
        return out, ct, nk

    def map_colors_batch(self, items, palettes, labels=False, ctx=None):
        """map_colors_mps of every pixel set in `items` to its own palette in `palettes`, in one call
        (dq_map_colors_batch_ctx).  Returns a list of outputs, each equal to map_colors_mps(items[i], palettes[i]) on the
        same context; with labels=True a list of (out, labels) pairs, labels = colortable_indexes(out, palettes[i])."""
        arrs = [_u32(a) for a in items]
        pals = [_u32(p) for p in palettes]
        if len(arrs) != len(pals):
            raise ValueError("one palette per item")
        if not arrs:
            return []
        offsets = np.zeros(len(arrs) + 1, np.uint32)
        np.cumsum([a.size for a in arrs], out=offsets[1:])
        flat = np.concatenate(arrs) if offsets[-1] else np.zeros(1, np.uint32)
        out = np.zeros_like(flat)
        lab = np.zeros_like(flat) if labels else None
        sizes = np.asarray([p.size for p in pals], np.int32)
        ct = np.concatenate(pals) if sizes.sum() else np.zeros(1, np.uint32)
        self.lib.dq_map_colors_batch_ctx(ctx or self.lib.dq_default_context(), len(arrs), _p(offsets), flat.size, _p(flat), _p(out),
                                         sizes.ctypes.data_as(C.POINTER(C.c_int)), _p(ct), _p(lab) if labels else None)
        outs = [out[offsets[i]:offsets[i + 1]].copy() for i in range(len(arrs))]
        if not labels:
            return outs
        return [(o, lab[offsets[i]:offsets[i + 1]].copy()) for i, o in enumerate(outs)]

    def map_colors_batch_device(self, flat, offsets, palettes, labels=False, ctx=None, out=None):
        """Device form (dq_map_colors_batch_device): `flat` is a CUDA tensor of 32-bit pixels holding the items end to
        end, item i = flat[offsets[i]:offsets[i+1]], mapped to palettes[i].  Returns (out tensor, labels tensor or None)."""
        import torch
        offs = _u32(offsets)
        pals = [_u32(p) for p in palettes]
        if offs.size != len(pals) + 1:
            raise ValueError("offsets need one entry more than palettes")
        if flat.dtype not in (torch.int32, torch.uint32) or not flat.is_cuda or not flat.is_contiguous():
            raise ValueError("flat must be a contiguous CUDA tensor of 32-bit pixels")
        out = torch.empty_like(flat) if out is None else out
        lab = torch.empty_like(flat) if labels else None
        sizes = np.asarray([p.size for p in pals], np.int32)
        ct = np.concatenate(pals) if sizes.sum() else np.zeros(1, np.uint32)
        if pals:
            torch.cuda.current_stream(flat.device).synchronize()  # the library works on its context's stream
            self.lib.dq_map_colors_batch_device(ctx or self.lib.dq_default_context(), len(pals), _p(offs), flat.numel(),
                                                flat.data_ptr(), out.data_ptr(), sizes.ctypes.data_as(C.POINTER(C.c_int)), _p(ct),
                                                lab.data_ptr() if labels else None)
        return out, lab

    def quant_regions(self, pixels, tags, ks, labels=False, ctx=None):
        """quant_recurse of every region of a tag image, each to its own palette, in one call (dq_quant_regions_ctx).
        Region r is pixels[tags == r] in raster order, quantized with ks[r] colours; pixels whose tag is >= len(ks) are
        in no region and come back as 0 (label 0).  Returns (out, palettes, actual_k[, labels]): palettes is the uint32
        array of sum(ks) words in which region r's palette starts at sum(ks[:r]) and holds actual_k[r] entries (0 for a
        region with no pixels); out[tags == r] and its palette equal quant_recurse_batch's result for that region."""
        px = _u32(pixels)
        tg = _u32(tags)
        nk = _u32(ks).copy()
        if tg.size != px.size:
            raise ValueError("one tag per pixel")
        out = np.zeros_like(px)
        lab = np.zeros_like(px) if labels else None
        ct = np.zeros(max(int(nk.astype(np.int64).sum()), 1), np.uint32)
        if nk.size:
            self.lib.dq_quant_regions_ctx(ctx or self.lib.dq_default_context(), px.size, _p(px), _p(tg), nk.size, _p(out), _p(nk),
                                          _p(ct), _p(lab) if labels else None)
        return (out, ct, nk, lab) if labels else (out, ct, nk)

    def quant_regions_device(self, pixels, tags, ks, labels=False, ctx=None, out=None, labels_out=None):
        """Device form (dq_quant_regions_device): `pixels` and `tags` are contiguous CUDA tensors of 32-bit words, one tag
        per pixel.  Writes out (and labels) at region pixels only: tensors passed as `out` / `labels_out` keep their other
        pixels (a `labels_out` tensor implies labels=True).  Returns (out, palettes, actual_k[, labels]) as quant_regions."""
        import torch
        nk = _u32(ks).copy()
        for t in (pixels, tags):
            if t.dtype not in (torch.int32, torch.uint32) or not t.is_cuda or not t.is_contiguous():
                raise ValueError("pixels and tags must be contiguous CUDA tensors of 32-bit words")
        if tags.numel() != pixels.numel():
            raise ValueError("one tag per pixel")
        labels = labels or labels_out is not None
        out = torch.zeros_like(pixels) if out is None else out
        lab = (torch.zeros_like(pixels) if labels_out is None else labels_out) if labels else None
        ct = np.zeros(max(int(nk.astype(np.int64).sum()), 1), np.uint32)
        if nk.size:
            torch.cuda.current_stream(pixels.device).synchronize()  # the library works on its context's stream
            self.lib.dq_quant_regions_device(ctx or self.lib.dq_default_context(), pixels.numel(), pixels.data_ptr(), tags.data_ptr(),
                                             nk.size, out.data_ptr(), _p(nk), _p(ct), lab.data_ptr() if labels else None)
        return (out, ct, nk, lab) if labels else (out, ct, nk)

    @staticmethod
    def _region_palettes(palettes, num_pixels, num_tags, labels):
        """(sizes, packed palettes) for dq_map_regions_*, after the checks the library would abort on."""
        if num_tags != num_pixels:
            raise ValueError("one tag per pixel")
        if len(palettes) > 1 << 24:
            raise ValueError(f"{len(palettes)} palettes; at most 2^24 regions")
        if any(np.ndim(p) != 1 for p in palettes):
            raise ValueError("one palette (a 1-D array, empty = not mapped) per region")
        pals = [_u32(p) for p in palettes]
        sizes = np.asarray([p.size for p in pals], np.int32)
        if labels and sizes.size and sizes.max() > 24000:
            raise ValueError("label images support palettes of at most 24000 entries")
        ct = np.concatenate(pals) if sizes.sum() else np.zeros(1, np.uint32)
        return sizes, ct

    def map_regions(self, pixels, tags, palettes, labels=False, ctx=None):
        """map_colors_mps of every region of a tag image, each to its own palette, in one call (dq_map_regions_ctx).
        Region r is pixels[tags == r] in raster order, mapped to palettes[r] (a uint32 array; an empty one leaves the
        region unmapped); pixels whose tag is >= len(palettes) are in no region.  Returns out, or (out, labels) with
        labels=True: out[tags == r] and its labels equal map_colors_batch's result for that region, and pixels in no
        region or in an unmapped region come back as 0."""
        px = _u32(pixels)
        tg = _u32(tags)
        sizes, ct = self._region_palettes(palettes, px.size, tg.size, labels)
        out = np.zeros_like(px)
        lab = np.zeros_like(px) if labels else None
        if sizes.size:
            self.lib.dq_map_regions_ctx(ctx or self.lib.dq_default_context(), px.size, _p(px), _p(tg), sizes.size,
                                        sizes.ctypes.data_as(C.POINTER(C.c_int)), _p(ct), _p(out), _p(lab) if labels else None)
        return (out, lab) if labels else out

    def map_regions_device(self, pixels, tags, palettes, labels=False, ctx=None, out=None, labels_out=None):
        """Device form (dq_map_regions_device): `pixels` and `tags` are contiguous CUDA tensors of 32-bit words, one tag
        per pixel.  Writes out (and labels) at the pixels of mapped regions only: tensors passed as `out` / `labels_out`
        keep their other pixels (a `labels_out` tensor implies labels=True).  Returns out, or (out, labels), as
        map_regions."""
        import torch
        for t in (pixels, tags):
            if t.dtype not in (torch.int32, torch.uint32) or not t.is_cuda or not t.is_contiguous():
                raise ValueError("pixels and tags must be contiguous CUDA tensors of 32-bit words")
        labels = labels or labels_out is not None
        sizes, ct = self._region_palettes(palettes, pixels.numel(), tags.numel(), labels)
        out = torch.zeros_like(pixels) if out is None else out
        lab = (torch.zeros_like(pixels) if labels_out is None else labels_out) if labels else None
        if sizes.size:
            torch.cuda.current_stream(pixels.device).synchronize()  # the library works on its context's stream
            self.lib.dq_map_regions_device(ctx or self.lib.dq_default_context(), pixels.numel(), pixels.data_ptr(), tags.data_ptr(),
                                           sizes.size, sizes.ctypes.data_as(C.POINTER(C.c_int)), _p(ct), out.data_ptr(),
                                           lab.data_ptr() if labels else None)
        return (out, lab) if labels else out

    def last_batch_stats(self, ctx=None):
        st = BatchStats()
        self.lib.dq_context_last_batch_stats(ctx or self.lib.dq_default_context(), C.byref(st))
        return st.as_dict()

    def map_colors_mps(self, pixels, colortable):
        px = _u32(pixels)
        ct = _u32(colortable).copy()
        out = np.zeros_like(px)
        self.lib.dq_map_colors_mps(_p(px), px.size, _p(out), _p(ct), ct.size)
        return out

    def calc_color_table(self, pixels, dec_factor=1, rows=1, cols=None):
        px = _u32(pixels)
        cols = px.size if cols is None else cols
        uniq = np.zeros(px.size, np.uint32)
        w = np.zeros(px.size, np.float64)
        n = C.c_int(0)
        rc = self.lib.dq_calc_color_table(_p(px), px.size, _p(uniq), rows, cols, dec_factor, C.byref(n), _p(w, _f64p))
        if rc != 0:
            return None
        return uniq[:n.value].copy(), w[:n.value].copy()

    def cut_bits(self, pixels, rbits, gbits, bbits):
        px = _u32(pixels)
        out = np.zeros_like(px)
        self.lib.dq_cut_bits(_p(px), px.size, _p(out), rbits, gbits, bbits)
        return out

    def srm_sorted_edges(self, image):
        """image: uint8 (height, width, channels>=3) interleaved.  Returns (n_pairs, 3) uint32: r1, r2, diff in the
        merge order of the reference's SRM (srm->ordered_pairs)."""
        im = np.ascontiguousarray(image, np.uint8)
        h, w, ch = im.shape
        n = self.lib.dq_srm_num_pairs(w, h)
        out = np.zeros((n, 3), np.uint32)
        self.lib.dq_srm_sorted_edges(im.ctypes.data, w, h, ch, w * ch, out.ctypes.data)
        return out

    def pixel_histogram(self, pixels):
        """generatePixelHistogram: (distinct 24-bit pixels ascending, counts)."""
        px = _u32(pixels)
        cap = min(px.size, 1 << 24)
        keys, counts = np.zeros(cap, np.uint32), np.zeros(cap, np.uint32)
        u = self.lib.dq_pixel_histogram(_p(px), px.size, _p(keys), _p(counts), cap)
        return keys[:u].copy(), counts[:u].copy()

    def block_vote(self, quant_pixels, width, height, dim=4):
        px = _u32(quant_pixels)
        bw, bh = -(-width // dim), -(-height // dim)
        out = np.zeros(bw * bh, np.uint32)
        self.lib.dq_block_vote(_p(px), width, height, dim, _p(out))
        return out.reshape(bh, bw)

    def quant_blocks(self, pixels, width, height, colortable, dim=4):
        """genHistogramsForBlocks' numeric part: remap to `colortable`, then one representative per block."""
        px = _u32(pixels)
        ct = _u32(colortable).copy()
        bw, bh = -(-width // dim), -(-height // dim)
        quant = np.zeros_like(px)
        blocks = np.zeros(bw * bh, np.uint32)
        self.lib.dq_quant_blocks(_p(px), width, height, dim, _p(ct), ct.size, _p(quant), _p(blocks))
        return quant, blocks.reshape(bh, bw)

    def colortable_indexes(self, quant_pixels, colortable, greyscale=False):
        """Label image: index of every quantized pixel in the caller's palette order (last duplicate wins)."""
        px = _u32(quant_pixels)
        ct = _u32(colortable).copy()
        out = np.zeros_like(px)
        self.lib.dq_colortable_indexes(_p(px), px.size, _p(ct), ct.size, _p(out), 1 if greyscale else 0)
        return out

    # -- host-only palette handling (no device) ------------------------------------------------
    def host_dedup_palette(self, colortable):
        ct = _u32(colortable).copy()
        n = self.lib.dq_host_dedup_palette(_p(ct), ct.size)
        return ct[:n].copy()

    def host_build_search_tables(self, colortable):
        ct = _u32(colortable).copy()
        srt = np.zeros_like(ct)
        lut = np.zeros(766, np.int32)
        self.lib.dq_host_build_search_tables(_p(ct), ct.size, _p(srt), lut.ctypes.data_as(C.POINTER(C.c_int32)))
        return srt, lut

    def host_build_label_table(self, colortable):
        """For each entry of host_build_search_tables' sorted palette, the index of the last entry of `colortable` with
        that 24-bit colour."""
        ct = _u32(colortable).copy()
        lab = np.zeros_like(ct)
        self.lib.dq_host_build_label_table(_p(ct), ct.size, _p(lab))
        return lab

    # -- diagnostics ---------------------------------------------------------------------------
    def last_stats(self, ctx=None):
        st = CallStats()
        self.lib.dq_context_last_stats(ctx or self.lib.dq_default_context(), C.byref(st))
        return st.as_dict()

    def histogram(self, pixels):
        px = _u32(pixels)
        col = np.zeros(px.size, np.uint32)
        cnt = np.zeros(px.size, np.uint32)
        u = self.lib.dq_debug_histogram(self.lib.dq_default_context(), _p(px), px.size, _p(col), _p(cnt))
        return col[:u].copy(), cnt[:u].copy()

    def split_points(self, colours, counts, norm, k, max_iters=10, num_bits=8):
        col = _u32(colours)
        cnt = _u32(counts)
        ct = np.zeros(max(int(k), 1), np.uint32)
        recs = (SplitRecord * max(int(k), 1))()
        means = np.zeros(3 * max(int(k), 1), np.float64)
        sizes = np.zeros(max(int(k), 1), np.uint32)
        n = self.lib.dq_debug_split_points(self.lib.dq_default_context(), _p(col), _p(cnt), col.size, norm, k, max_iters,
                                           num_bits, _p(ct), recs, _p(means, _f64p), _p(sizes))
        return ct[:n].copy(), [recs[i] for i in range(max(int(k) - 1, 0))], means.reshape(-1, 3), sizes


class FramePipeline:
    """dq_pipeline: quant_recurse over a stream of frames, `depth` frames (lanes) in flight on one GPU."""

    def __init__(self, lib, device, max_pixels, depth=3, split_ctas=0):
        self.lib = lib
        self.handle = lib.dq_pipeline_create_lanes(device, max_pixels, depth, split_ctas)
        self._keep = []

    def submit(self, pixels, out, k, colortable, nk, all_unique=0):
        """pixels/out/colortable: uint32 numpy arrays (or objects exposing .ctypes) that outlive flush();
        nk: ctypes.c_uint32 holding the requested K (updated in place).  Returns the frame's ticket."""
        self._keep.append((pixels, out, colortable, nk))
        return self.lib.dq_pipeline_submit(self.handle, pixels.size, _p(pixels), _p(out), C.byref(nk), _p(colortable), all_unique)

    def submit_device(self, d_in, d_out, num_pixels, colortable, nk, all_unique=0):
        """d_in/d_out: device addresses (ints) of uint32 frames on the pipeline's GPU."""
        self._keep.append((colortable, nk))
        return self.lib.dq_pipeline_submit_device(self.handle, num_pixels, d_in, d_out, C.byref(nk), _p(colortable), all_unique)

    def wait(self, ticket):
        self.lib.dq_pipeline_wait(self.handle, ticket)

    def flush(self):
        self.lib.dq_pipeline_flush(self.handle)
        self._keep.clear()
        return float(self.lib.dq_pipeline_last_elapsed_ms(self.handle))

    def close(self):
        if self.handle:
            self.lib.dq_pipeline_destroy(self.handle)
            self.handle = None


# ---- multi-GPU partitioning (host logic; BASELINE.json configs 3 and 4, SURVEY.md 8e) -------------------
def frames_for_rank(num_frames, world_size, rank):
    """Frame sharding: contiguous blocks, sizes differ by at most one, no collective on the data path."""
    base, extra = divmod(num_frames, world_size)
    start = rank * base + min(rank, extra)
    return range(start, start + base + (1 if rank < extra else 0))


def rows_for_rank(height, world_size, rank):
    """Pixel-row sharding of one image: contiguous row blocks (sizes differ by at most one)."""
    r = frames_for_rank(height, world_size, rank)
    return r.start, r.stop


def merge_histograms(colour_lists, count_lists):
    """Exact merge of per-shard (colour, count) lists: counts are additive, so the merged histogram -- and
    every sum the divisive phase takes over it -- is independent of the number of shards."""
    colours = np.concatenate([np.asarray(c, np.uint32) for c in colour_lists])
    counts = np.concatenate([np.asarray(c, np.uint64) for c in count_lists])
    uniq, inv = np.unique(colours, return_inverse=True)
    merged = np.zeros(uniq.size, np.uint64)
    np.add.at(merged, inv, counts)
    return uniq, merged


class RowShards:
    """dq_rows: quant_recurse of ONE image whose pixel rows are spread over the ranks of a torch.distributed group, the
    exchange (one grouped ncclAllGather per image) inside the library.  torch.distributed only carries the 128-byte NCCL
    id from rank 0 to the others when the object is created."""

    def __init__(self, lib, ctx, dist=None, list_capacity=1 << 18):
        import torch
        self.lib, self.ctx = lib, ctx
        world = dist.get_world_size() if dist is not None else 1
        rank = dist.get_rank() if dist is not None else 0
        ident = (C.c_ubyte * 128)()
        if world > 1:
            if rank == 0:
                lib.dq_rows_unique_id(ident)
            t = torch.tensor(list(ident), dtype=torch.uint8, device="cuda")
            dist.broadcast(t, 0)
            ident = (C.c_ubyte * 128)(*t.cpu().tolist())
        self.handle = lib.dq_rows_create(ctx, world, rank, ident, list_capacity)

    def quant_recurse(self, shard, total_pixels, k, out=None):
        """shard: this rank's rows as a flat CUDA int32 tensor.  Returns (out_shard, palette)."""
        import torch
        out = torch.empty_like(shard) if out is None else out
        ct = np.zeros(max(int(k), 1), np.uint32)
        nk = C.c_uint32(k)
        self.lib.dq_rows_quant_recurse(self.handle, shard.data_ptr(), shard.numel(), total_pixels, out.data_ptr(), C.byref(nk), _p(ct))
        return out, ct[:nk.value].copy()

    def close(self):
        if self.handle:
            self.lib.dq_rows_destroy(self.handle)
            self.handle = None
