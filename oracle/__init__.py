"""oracle/ -- TEST INFRASTRUCTURE ONLY.

ctypes bindings for the two CPU checkers:

* ``Oracle``    -> oracle/libdivquant_oracle.so, this repo's restatement (divquant_oracle.cpp).
* ``Reference`` -> oracle/_ref/libdivquant_ref.so, the UNMODIFIED reference sources compiled from
                   /root/reference by oracle/Makefile (present only where it was built).

Only tests/, ``__graft_entry__.smoke()`` and bench.py's ``cpu_baseline`` / ``--impl reference``
legs may import this package, and only as the checker.  The product never does.
"""
import contextlib
import ctypes as C
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(_HERE, "libdivquant_oracle.so")
REF_SO = os.path.join(_HERE, "_ref", "libdivquant_ref.so")

_u32p = C.POINTER(C.c_uint32)
_i32p = C.POINTER(C.c_int32)
_f64p = C.POINTER(C.c_double)


def build(quiet=True):
    """Compile the restatement and, when /root/reference is mounted, the reference itself."""
    subprocess.run(["make", "-C", _HERE, "all"], check=True,
                   stdout=subprocess.DEVNULL if quiet else None)


@contextlib.contextmanager
def muted(fds=(1, 2)):
    """Silence C-level stdout/stderr (the reference prints timing lines and '# empty clusters')."""
    sys.stdout.flush()
    sys.stderr.flush()
    saved = [(fd, os.dup(fd)) for fd in fds]
    null = os.open(os.devnull, os.O_WRONLY)
    try:
        for fd in fds:
            os.dup2(null, fd)
        yield
    finally:
        C.CDLL(None).fflush(None)
        for fd, keep in saved:
            os.dup2(keep, fd)
            os.close(keep)
        os.close(null)


def _ptr(a, t=_u32p):
    return a.ctypes.data_as(t)


def _u32(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.uint32).ravel())


class SplitRecord(C.Structure):
    _fields_ = [("new_index", C.c_int32), ("old_index", C.c_int32), ("cut_axis", C.c_int32),
                ("num_points", C.c_int32), ("new_size", C.c_int32), ("is_last", C.c_int32),
                ("cut_pos", C.c_double), ("total_weight", C.c_double), ("new_weight", C.c_double),
                ("old_weight", C.c_double), ("new_mean", C.c_double * 3), ("old_mean", C.c_double * 3),
                ("new_var", C.c_double * 3), ("old_var", C.c_double * 3), ("new_tse", C.c_double),
                ("old_tse", C.c_double)]


class Oracle:
    """The restatement.  Method names follow the reference entry points they restate."""

    def __init__(self, path=ORACLE_SO):
        if not os.path.exists(path):
            build()
        self.lib = C.CDLL(path)
        L = self.lib
        L.oracle_calc_color_table.restype = C.c_int
        L.oracle_calc_color_table.argtypes = [_u32p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, _u32p, _f64p, _u32p]
        L.oracle_cut_bits.restype = C.c_int
        L.oracle_cut_bits.argtypes = [_u32p, C.c_uint32, _u32p, C.c_int, C.c_int, C.c_int]
        L.oracle_quant_varpart_fast.restype = C.c_int
        L.oracle_quant_varpart_fast.argtypes = [C.c_uint32, _u32p, C.c_uint32, C.c_uint32, _u32p, _u32p, C.c_int,
                                                C.c_int, C.c_int, C.c_int, C.POINTER(SplitRecord), _i32p]
        L.oracle_quant_varpart_fast_exact.restype = C.c_int
        L.oracle_quant_varpart_fast_exact.argtypes = L.oracle_quant_varpart_fast.argtypes
        L.oracle_map_colors_mps.restype = None
        L.oracle_map_colors_mps.argtypes = [_u32p, C.c_uint32, _u32p, _u32p, C.c_int]
        L.oracle_map_colors_bruteforce.restype = None
        L.oracle_map_colors_bruteforce.argtypes = [_u32p, C.c_uint32, _u32p, _u32p, C.c_int]
        L.oracle_build_search_tables.restype = None
        L.oracle_build_search_tables.argtypes = [_u32p, C.c_int, _u32p, _i32p]
        L.oracle_quant_recurse.restype = None
        L.oracle_quant_recurse.argtypes = [C.c_uint32, _u32p, _u32p, _u32p, _u32p, C.c_int]
        L.oracle_colortable_indexes.restype = C.c_int
        L.oracle_colortable_indexes.argtypes = [_u32p, C.c_uint32, _u32p, C.c_int, _u32p]
        L.oracle_block_vote.restype = None
        L.oracle_block_vote.argtypes = [_u32p, C.c_uint32, C.c_uint32, C.c_uint32, _u32p]
        L.oracle_srm_sorted_edges.restype = C.c_uint32
        L.oracle_srm_sorted_edges.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, _u32p]
        L.oracle_hash_words.restype = C.c_uint64
        L.oracle_hash_words.argtypes = [_u32p, C.c_uint64]
        L.oracle_generate.restype = None
        L.oracle_generate.argtypes = [C.c_int, C.c_uint32, C.c_uint32, C.c_uint64, _u32p]

    # -- histogram ------------------------------------------------------------------------
    def calc_color_table(self, pixels, dec_factor=1, rows=1, cols=None):
        px = _u32(pixels)
        cols = px.size if cols is None else cols
        uniq = np.empty(px.size, np.uint32)
        w = np.empty(px.size, np.float64)
        cnt = np.empty(px.size, np.uint32)
        u = self.lib.oracle_calc_color_table(_ptr(px), px.size, rows, cols, dec_factor, _ptr(uniq),
                                             _ptr(w, _f64p), _ptr(cnt))
        if u < 0:
            return None
        return uniq[:u].copy(), w[:u].copy(), cnt[:u].copy()

    def cut_bits(self, pixels, rbits, gbits, bbits):
        px = _u32(pixels)
        out = np.zeros_like(px)
        ok = self.lib.oracle_cut_bits(_ptr(px), px.size, _ptr(out), rbits, gbits, bbits)
        return out if ok else None

    # -- quantize -------------------------------------------------------------------------
    def quant_varpart_resolved(self, pixels, k, num_bits=8, dec_factor=1, max_iters=10, rows=1, cols=None):
        """CPU model of the device's DEFAULT large-input path: exact integer sums + tie audit + the resolver (palette
        roundings and cuts settled by the reference's own mean of the node, csrc/dq_resolve.cu).  Returns (palette,
        info) with info = {"left": decisions still flagged (axis / hyperplane / TSE), "roundings": ..., "cuts_confirmed": ...,
        "cuts_forced": ...}; with left == 0 the palette must be the reference's.  rows / cols: the sampling grid of
        calc_color_table, as in quant_varpart_fast."""
        px = _u32(pixels)
        cols = px.size if cols is None else cols
        ct = np.zeros(max(k, 1), np.uint32)
        nk = C.c_uint32(k)
        flags = np.zeros(9, np.uint32)
        fn = self.lib.oracle_quant_varpart_fast_exact_resolved
        fn.restype = C.c_int
        fn.argtypes = [C.c_uint32, _u32p, C.c_uint32, C.c_uint32, _u32p, _u32p, C.c_int, C.c_int, C.c_int, C.c_int, _u32p]
        fn(px.size, _ptr(px), rows, cols, C.byref(nk), _ptr(ct), num_bits, dec_factor, max_iters, 0, _ptr(flags))
        return ct[:nk.value].copy(), {"left": int(flags[0]), "roundings": int(flags[6]), "cuts_confirmed": int(flags[7]),
                                      "cuts_forced": int(flags[8]), "left_axis": int(flags[1]), "left_hyperplane": int(flags[3]),
                                      "left_tse": int(flags[4])}

    def quant_varpart_fast(self, pixels, k, num_bits=8, dec_factor=1, max_iters=10, all_unique=0,
                           with_records=False, exact_counts=False, rows=1, cols=None):
        px = _u32(pixels)
        cols = px.size if cols is None else cols
        ct = np.zeros(max(k, 1), np.uint32)
        nk = C.c_uint32(k)
        recs = (SplitRecord * max(k, 1))()
        nrec = C.c_int32(0)
        fn = self.lib.oracle_quant_varpart_fast_exact if exact_counts else self.lib.oracle_quant_varpart_fast
        empty = fn(px.size, _ptr(px), rows, cols, C.byref(nk), _ptr(ct), num_bits,
                   dec_factor, max_iters, all_unique, recs, C.byref(nrec))
        pal = ct[:nk.value].copy()
        if with_records:
            return pal, empty, [recs[i] for i in range(nrec.value)]
        return pal, empty

    def quant_recurse(self, pixels, k, all_unique=0):
        px = _u32(pixels)
        out = np.zeros_like(px)
        ct = np.zeros(max(k, 1), np.uint32)
        nk = C.c_uint32(k)
        self.lib.oracle_quant_recurse(px.size, _ptr(px), _ptr(out), C.byref(nk), _ptr(ct), all_unique)
        return out, ct[:nk.value].copy()

    # -- remap ----------------------------------------------------------------------------
    def map_colors_mps(self, pixels, colortable, bruteforce=False):
        px = _u32(pixels)
        ct = _u32(colortable).copy()
        out = np.zeros_like(px)
        fn = self.lib.oracle_map_colors_bruteforce if bruteforce else self.lib.oracle_map_colors_mps
        fn(_ptr(px), px.size, _ptr(out), _ptr(ct), ct.size)
        return out

    def build_search_tables(self, colortable):
        ct = _u32(colortable).copy()
        srt = np.zeros_like(ct)
        lut = np.zeros(766, np.int32)
        self.lib.oracle_build_search_tables(_ptr(ct), ct.size, _ptr(srt), _ptr(lut, _i32p))
        return srt, lut

    def colortable_indexes(self, quant_pixels, colortable):
        px = _u32(quant_pixels)
        ct = _u32(colortable).copy()
        out = np.zeros_like(px)
        rc = self.lib.oracle_colortable_indexes(_ptr(px), px.size, _ptr(ct), ct.size, _ptr(out))
        if rc != 0:
            raise ValueError("pixel not present in colortable")
        return out

    def block_vote(self, quant_pixels, width, height, dim=4):
        px = _u32(quant_pixels)
        bw, bh = -(-width // dim), -(-height // dim)
        out = np.zeros(bw * bh, np.uint32)
        self.lib.oracle_block_vote(_ptr(px), width, height, dim, _ptr(out))
        return out.reshape(bh, bw)

    def srm_sorted_edges(self, image):
        """image: uint8 array (height, width, channels) in B,G,R[,A] order.  Returns (n_pairs, 3) uint32: r1, r2, diff."""
        im = np.ascontiguousarray(image, np.uint8)
        h, w, ch = im.shape
        n = self.lib.oracle_srm_sorted_edges(im.ctypes.data, w, h, ch, w * ch, None)
        out = np.zeros((n, 3), np.uint32)
        self.lib.oracle_srm_sorted_edges(im.ctypes.data, w, h, ch, w * ch, _ptr(out.reshape(-1)))
        return out

    # -- utilities ------------------------------------------------------------------------
    def hash_words(self, words):
        w = _u32(words)
        return int(self.lib.oracle_hash_words(_ptr(w), w.size))

    def generate(self, kind, width, height, seed=12345):
        out = np.empty(width * height, np.uint32)
        self.lib.oracle_generate(kind, width, height, seed, _ptr(out))
        return out


SRM_REF_SO = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "libsrm_ref.so")


class ReferenceSRM:
    """The unmodified reference SRM (oracle/_ref/libsrm_ref.so): its sorted edge list and its segmentation."""

    def __init__(self, path=SRM_REF_SO):
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.lib = C.CDLL(path)
        self.lib.ref_srm_sorted_edges.restype = C.c_uint
        self.lib.ref_srm_sorted_edges.argtypes = [C.c_double, C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p, _u32p]

    def run_with_pairs(self, image, pairs, q=128.0):
        """The reference's SRM (initialize, union-find merge loop srm.c:179-190, merge_small_regions, finalize) driven by a
        SUPPLIED sorted edge list (n_pairs, 3) uint32 instead of the one segmentation() builds.  Returns the segmented image."""
        im = np.ascontiguousarray(image, np.uint8).copy()
        h, w, ch = im.shape
        out_img = np.zeros_like(im)
        pr = np.ascontiguousarray(pairs, np.uint32)
        fn = self.lib.ref_srm_run_with_pairs
        fn.restype = None
        fn.argtypes = [C.c_double, C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p, _u32p]
        fn(q, w, h, ch, w * ch, im.ctypes.data, out_img.ctypes.data, _ptr(pr.reshape(-1)))
        return out_img

    def sorted_edges(self, image, q=32.0):
        im = np.ascontiguousarray(image, np.uint8).copy()
        h, w, ch = im.shape
        out_img = np.zeros_like(im)
        n = self.lib.ref_srm_sorted_edges(q, w, h, ch, w * ch, im.ctypes.data, out_img.ctypes.data, None)
        pairs = np.zeros((n, 3), np.uint32)
        self.lib.ref_srm_sorted_edges(q, w, h, ch, w * ch, im.ctypes.data, out_img.ctypes.data, _ptr(pairs.reshape(-1)))
        return pairs, out_img


class Reference:
    """The unmodified reference build (oracle/_ref).  Prints the reference's own timing lines."""

    def __init__(self, path=REF_SO):
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.lib = C.CDLL(path)
        L = self.lib
        L.ref_quant_recurse.restype = None
        L.ref_quant_recurse.argtypes = [C.c_uint32, _u32p, _u32p, _u32p, _u32p, C.c_int]
        L.ref_quant_varpart_fast.restype = None
        L.ref_quant_varpart_fast.argtypes = [C.c_uint32, _u32p, _u32p, C.c_uint32, C.c_uint32, _u32p, _u32p, C.c_int,
                                             C.c_int, C.c_int, C.c_int]
        L.ref_map_colors_mps.restype = None
        L.ref_map_colors_mps.argtypes = [_u32p, C.c_uint32, _u32p, _u32p, C.c_int]
        L.ref_calc_color_table.restype = C.c_int
        L.ref_calc_color_table.argtypes = [_u32p, C.c_uint32, _u32p, C.c_uint32, C.c_uint32, C.c_int, _f64p]
        L.ref_cut_bits.restype = None
        L.ref_cut_bits.argtypes = [_u32p, C.c_uint32, _u32p, C.c_int, C.c_int, C.c_int]

    @staticmethod
    def available():
        return os.path.exists(REF_SO)

    def quant_recurse(self, pixels, k, all_unique=0):
        px = _u32(pixels)
        out = np.zeros_like(px)
        ct = np.zeros(max(k, 1), np.uint32)
        nk = C.c_uint32(k)
        with muted():
            self.lib.ref_quant_recurse(px.size, _ptr(px), _ptr(out), C.byref(nk), _ptr(ct), all_unique)
        return out, ct[:nk.value].copy()

    def quant_varpart_fast(self, pixels, k, num_bits=8, dec_factor=1, max_iters=10, all_unique=0):
        px = _u32(pixels)
        tmp = np.zeros_like(px)
        ct = np.zeros(max(k, 1), np.uint32)
        nk = C.c_uint32(k)
        with muted():
            self.lib.ref_quant_varpart_fast(px.size, _ptr(px), _ptr(tmp), 1, px.size, C.byref(nk), _ptr(ct),
                                            num_bits, dec_factor, max_iters, all_unique)
        return ct[:nk.value].copy(), k - nk.value

    def map_colors_mps(self, pixels, colortable):
        px = _u32(pixels)
        ct = _u32(colortable).copy()
        out = np.zeros_like(px)
        self.lib.ref_map_colors_mps(_ptr(px), px.size, _ptr(out), _ptr(ct), ct.size)
        return out

    def calc_color_table(self, pixels, dec_factor=1, rows=1, cols=None):
        px = _u32(pixels)
        cols = px.size if cols is None else cols
        uniq = np.empty(px.size, np.uint32)
        w = np.empty(px.size, np.float64)
        u = self.lib.ref_calc_color_table(_ptr(px), px.size, _ptr(uniq), rows, cols, dec_factor, _ptr(w, _f64p))
        if u < 0:
            return None
        return uniq[:u].copy(), w[:u].copy()

    def cut_bits(self, pixels, rbits, gbits, bbits):
        px = _u32(pixels)
        out = np.zeros_like(px)
        self.lib.ref_cut_bits(_ptr(px), px.size, _ptr(out), rbits, gbits, bbits)
        return out
