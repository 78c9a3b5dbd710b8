"""GPU parity tests: the CUDA path, called through the C ABI (ctypes on libdivquant_b200.so), against
the oracle, the committed golden fixtures of the compiled reference, and size-independent properties.

Parity bar (BASELINE.json north_star):
  * integer work (histogram, unique-colour set, remap / label image): bit-exact;
  * uniform-weight quantisation (allPixelsUnique=1): bit-exact, the reference itself is integer-exact there;
  * weighted quantisation: palettes bit-exact on every named config; in general bit-exact against the
    oracle's exact-count model, split statistics within REL_TOL = 1e-6 of the reference restatement.
"""
import numpy as np
import pytest

from oracle import muted
from conftest import small_case_ids

pytestmark = pytest.mark.gpu
import os as _os
ROOT_DIR = _os.path.dirname(_os.path.dirname(_os.path.abspath(__file__)))
REL_TOL = 1e-6  # north_star: "split statistics within 1e-6 relative"


def test_kats_through_c_abi(dq, kats):
    for kat in kats:
        px = np.array(kat["pixels"], np.uint32)
        for uq in (1, 0):
            with muted((2,)):
                out, pal = dq.quant_recurse(px, kat["k"], uq)
            assert [int(x) for x in pal] == kat["palette"], (kat["name"], uq)
            assert [int(x) for x in out] == kat["out_pixels"], (kat["name"], uq)


def test_histogram_bit_exact(dq, oracle):
    rng = np.random.default_rng(1)
    for n in (1, 2, 3, 4, 5, 31, 32, 33, 127, 1000, 4099, 200001):
        px = rng.integers(0, 1 << 24, n, dtype=np.uint32)
        px[:: max(1, n // 7)] = px[0]
        px |= np.uint32(0xFF000000) * rng.integers(0, 2, n, dtype=np.uint32)
        col, cnt = dq.histogram(px)
        uc, ucnt = np.unique(px & 0xFFFFFF, return_counts=True)
        order = np.argsort(col)
        assert np.array_equal(col[order], uc) and np.array_equal(cnt[order], ucnt.astype(np.uint32)), n
    # the direct table must be clean again: a second, different histogram is still exact
    px = rng.integers(0, 64, 5000, dtype=np.uint32)
    col, cnt = dq.histogram(px)
    assert cnt.sum() == 5000 and col.size == np.unique(px).size


def test_calc_color_table_order_and_weights(dq, oracle):
    rng = np.random.default_rng(8)
    for n, dec in ((1, 1), (17, 1), (5000, 1), (5000, 2), (5003, 3), (70000, 1)):
        base = rng.integers(0, 1 << 24, max(1, n // 5), dtype=np.uint32)
        px = base[rng.integers(0, base.size, n)] | np.uint32(0xFF000000)
        col, w = dq.calc_color_table(px, dec)
        ocol, ow, _ = oracle.calc_color_table(px, dec)
        assert np.array_equal(col, ocol), (n, dec)  # hash-bucket order, most recently first-seen first
        assert np.array_equal(w, ow), (n, dec)      # bit-exact doubles: norm * count


def test_cut_bits(dq, oracle):
    rng = np.random.default_rng(4)
    px = rng.integers(0, 1 << 32, 10007, dtype=np.uint64).astype(np.uint32)
    for bits in ((8, 8, 8), (5, 5, 5), (1, 1, 1), (7, 5, 3), (8, 1, 4)):
        assert np.array_equal(dq.cut_bits(px, *bits), oracle.cut_bits(px, *bits)), bits
    with muted((2,)):
        assert np.array_equal(dq.cut_bits(px, 0, 8, 8), np.zeros_like(px))  # rejected: message, no output


def test_small_cases_uniform_path_bit_exact_vs_reference(dq, golden):
    for i in small_case_ids(golden):
        px, k = golden[f"small{i}_in"], int(golden[f"small{i}_k"][0])
        with muted((2,)):
            out, pal = dq.quant_recurse(px, k, 1)
        assert np.array_equal(pal, golden[f"small{i}_u1_palette"]), i
        assert np.array_equal(out, golden[f"small{i}_u1_out"]), i


# Up to this many unique colours the tests demand the reference's result bit for bit on EVERY input, ties included: the
# ordered path sums in the reference's order up to its default limit (4096, kExactDefaultPoints in csrc/dq_split.cuh);
# above it the exact-integer kernels run with the tie audit, and flagged frames are settled by the resolver or re-run on
# the ordered path (which takes up to 262 144 colours).
EXACT_MAX_POINTS = 65536
EXACT_DEFAULT_LIMIT = 4096


def test_small_cases_weighted_path(dq, oracle, golden):
    """Weighted path (allPixelsUnique=0).  Up to EXACT_MAX_POINTS unique colours the device reproduces the
    reference's sequential double sums, so the result is the reference's bit for bit -- ties included.  Larger
    inputs use exact integer sums: bit-exact against the oracle's exact-count model always, and against the
    reference unless a decision sits exactly on a tie (none of the named configs does)."""
    ids = small_case_ids(golden)
    small = large_agree = large = 0
    for i in ids:
        px, k = golden[f"small{i}_in"], int(golden[f"small{i}_k"][0])
        u = np.unique(px & 0xFFFFFF).size
        with muted((2,)):
            pal, empty = dq.quant_varpart_fast(px, k)
            out, pal2 = dq.quant_recurse(px, k, 0)
        ref_pal = golden[f"small{i}_u0_palette"]
        if u <= EXACT_MAX_POINTS and k <= 4096:
            small += 1
            with muted():
                ref_vp, ref_empty = oracle.quant_varpart_fast(px, k)
            assert np.array_equal(pal, ref_vp) and empty == ref_empty, (i, u, k)
            assert np.array_equal(pal2, ref_pal), (i, u, k)
            assert np.array_equal(out, golden[f"small{i}_u0_out"]), (i, u, k)
            continue
        large += 1
        with muted():
            model, mempty = oracle.quant_varpart_fast(px, k, exact_counts=True)
        assert np.array_equal(pal, model) and empty == mempty, i
        if np.array_equal(pal2, ref_pal):
            large_agree += 1
            assert np.array_equal(out, golden[f"small{i}_u0_out"]), i
        else:
            assert np.array_equal(out, oracle.map_colors_mps(px, pal2)), i
    assert small >= 10
    assert large_agree >= large // 2


def test_tie_heavy_inputs_match_reference_order(dq, oracle):
    """Inputs built to sit on ties (few colours, equal counts, symmetric layouts, K > U, bits cut, decimation):
    the reference resolves them by the rounding noise of its sequential sums in calc_color_table order."""
    rng = np.random.default_rng(77)
    cases = []
    for t in range(40):
        ncol = int(rng.integers(2, 40))
        base = rng.integers(0, 256, (ncol, 3))
        if t % 3 == 0:  # symmetric around the centre of the cube
            base = np.concatenate([base, 255 - base])
        pal = ((base[:, 0] << 16) | (base[:, 1] << 8) | base[:, 2]).astype(np.uint32)
        reps = int(rng.integers(1, 5))
        px = np.tile(pal, reps) if t % 2 == 0 else pal[rng.integers(0, pal.size, pal.size * reps)]
        px = px | np.uint32(0xFF000000 if t % 4 else 0)
        cases.append((px, int(rng.choice([2, 3, 4, 8, 16, 64, 256]))))
    checker = np.indices((16, 16)).sum(axis=0) % 2
    cases.append((np.where(checker.ravel() == 1, 0x00FFFFFF, 0).astype(np.uint32), 2))
    cases.append((np.where(checker.ravel() == 1, 0x00FF0000, 0x000000FF).astype(np.uint32), 4))
    grey = (np.arange(256, dtype=np.uint32) * 0x010101)
    cases.append((np.concatenate([grey, grey[::-1]]), 16))
    for n, (px, k) in enumerate(cases):
        with muted():
            ref_out, ref_pal = oracle.quant_recurse(px, k, 0)
            ref_vp, ref_empty = oracle.quant_varpart_fast(px, k)
        with muted((2,)):
            out, pal = dq.quant_recurse(px, k, 0)
            vp, empty = dq.quant_varpart_fast(px, k)
        assert np.array_equal(pal, ref_pal), (n, k, px.size)
        assert np.array_equal(out, ref_out), (n, k, px.size)
        assert np.array_equal(vp, ref_vp) and empty == ref_empty, (n, k)
    # bits cut and decimation go through the same histogram -> same ordering rules
    px = cases[0][0]
    px = np.tile(px, 8)[:240]
    for bits, dec, rows, cols in ((5, 1, 1, 240), (8, 2, 12, 20), (6, 3, 12, 20)):
        with muted():
            ref_vp, ref_empty = oracle.quant_varpart_fast(px, 8, num_bits=bits, dec_factor=dec, rows=rows, cols=cols)
        with muted((2,)):
            vp, empty = dq.quant_varpart_fast(px, 8, num_bits=bits, dec_factor=dec, rows=rows, cols=cols)
        assert np.array_equal(vp, ref_vp) and empty == ref_empty, (bits, dec)


PALETTE_TOL_LSB = 1  # north_star: "refined palette entries within 1 LSB per channel after rounding"


def test_natural_crops_ordered_and_integer_paths(dq, oracle, golden):
    """36 seeded crops of Batman / Cookie / G1 (tests/golden/make_golden.py: crop_specs; 4 000 .. 60 000 unique colours),
    palettes and image fingerprints from the compiled reference.
    * Default (ordered path up to EXACT_MAX_POINTS colours): bit-identical palette and mapped image, every crop.
    * Ordered path off -> the exact-integer kernels, i.e. what inputs ABOVE the limit get: a decision that sits EXACTLY on
      a tie can come out differently -- in practice the final `(uint8)(mean + 0.5)` of a small cluster whose mean is
      x.5.  The bar there is north_star's floating-point tolerance: every palette entry within PALETTE_TOL_LSB per
      channel; where the palettes are equal the mapped image is bit-exact.  Measured on these 36 crops: 23 bit-identical,
      10 with a few entries off by one LSB, 3 where a tie changes which cluster is split (crops with few colours and
      K = 256, i.e. tiny clusters -- the regime the ordered path exists for).  The thresholds below pin that."""
    import sys
    sys.path.insert(0, _os.path.join(ROOT_DIR, "tests", "golden"))
    from make_golden import crop_pixels
    shaped = {}
    for name in ("batman", "cookie"):
        z = np.load(_os.path.join(ROOT_DIR, "tests", "golden", f"{name}_px.npz"))
        shaped[name] = z["px"].reshape(int(z["shape"][0]), int(z["shape"][1]))
    shaped["g1"] = oracle.generate(1, 1920, 1080, 99).reshape(1080, 1920)
    specs = golden["crop_specs"]
    ctx = dq.lib.dq_default_context()
    for ordered in (1, 0):
        dq.lib.dq_context_set_exact_small(ctx, ordered)
        identical = within_tol = structural = 0
        try:
            for i, spec in enumerate(specs):
                px = crop_pixels(shaped, spec)
                ref_pal = golden[f"crop{i}_palette"]
                with muted((2,)):
                    out, pal = dq.quant_recurse(px, int(spec[6]), 0)
                if np.array_equal(pal, ref_pal):
                    identical += 1
                    assert oracle.hash_words(out) == int(golden[f"crop{i}_out_hash"][0]), i   # integer work: bit-exact
                    continue
                assert not (ordered and int(golden[f"crop{i}_unique"][0]) <= EXACT_MAX_POINTS), (i, "ordered path must be identical")
                # the tie audit's contract: a frame the exact-integer kernels get wrong is a frame they flagged
                assert dq.last_stats()["tie_flags"] != 0, (i, "integer path differs from the reference without a tie flag")
                assert np.array_equal(out, oracle.map_colors_mps(px, pal)), i                 # remap of OUR palette: bit-exact
                if pal.size == ref_pal.size:
                    sh = np.array([16, 8, 0])
                    d = np.abs(((pal[:, None] >> sh) & 0xFF).astype(int) - ((ref_pal[:, None] >> sh) & 0xFF).astype(int)).max()
                    if d <= PALETTE_TOL_LSB:
                        within_tol += 1
                        continue
                structural += 1
        finally:
            dq.lib.dq_context_set_exact_small(ctx, 1)
        assert identical + within_tol + structural == len(specs)
        if ordered:
            assert identical == len(specs), (identical, within_tol, structural)
        else:
            assert identical >= 20, (identical, within_tol, structural)
            assert structural <= 4, (identical, within_tol, structural)


def test_map_colors_random_palettes(dq, oracle, golden):
    rng = np.random.default_rng(6)
    for i in small_case_ids(golden):
        assert np.array_equal(dq.map_colors_mps(golden[f"small{i}_in"], golden[f"small{i}_mappal"]), golden[f"small{i}_mapout"])
    for trial in range(12):
        n = int(rng.integers(1, 300000))
        px = rng.integers(0, 1 << 24, n, dtype=np.uint32)
        if trial % 2:  # few colours repeated often -> the unique-colour table path
            base = rng.integers(0, 1 << 24, 500, dtype=np.uint32)
            px = base[rng.integers(0, base.size, n)]
        k = int(rng.choice([1, 2, 7, 64, 125, 256, 257, 1000]))
        pal = rng.integers(0, 1 << 24, k, dtype=np.uint32)
        if trial % 3 == 0:
            pal[rng.integers(0, k, k // 3 + 1)] = pal[0]
        assert np.array_equal(dq.map_colors_mps(px, pal), oracle.map_colors_mps(px, pal)), (trial, n, k)


def test_map_colors_grid125_ties(dq, oracle, golden):
    # equal channel sums everywhere: the observable part of std::sort's permutation (SURVEY.md 7)
    r, g, b = np.meshgrid(np.arange(0, 256, 3), np.arange(0, 256, 5), np.arange(0, 256, 5), indexing="ij")
    px = ((r.astype(np.uint32) << 16) | (g.astype(np.uint32) << 8) | b.astype(np.uint32)).ravel()
    assert np.array_equal(dq.map_colors_mps(px, golden["grid125"]), oracle.map_colors_mps(px, golden["grid125"]))


@pytest.mark.parametrize("name", ["batman", "cookie"])
def test_fixture_images_bit_exact_vs_reference(dq, oracle, golden, images, name):
    px = images[name]
    for k in (4, 64, 125, 256):
        out, pal = dq.quant_recurse(px, k, 0)
        assert np.array_equal(pal, golden[f"{name}_k{k}_palette"]), k
        assert oracle.hash_words(out) == int(golden[f"{name}_k{k}_out_hash"][0]), k
    out = dq.map_colors_mps(px, golden["grid125"])
    assert oracle.hash_words(out) == int(golden[f"{name}_grid125_out_hash"][0])
    # label image consumed downstream (OpenCVUtil.cpp:787-849): index into the caller's palette
    labels = oracle.colortable_indexes(out[:5000], golden["grid125"])
    assert np.array_equal(golden["grid125"][labels] & 0xFFFFFF, out[:5000])


@pytest.mark.parametrize("tag,kind,w,h,k", [("g1_1080_k256", 1, 1920, 1080, 256), ("g1_1080_k64", 1, 1920, 1080, 64),
                                           ("g1_4k_k256", 1, 3840, 2160, 256), ("g2_640x360_k256", 2, 640, 360, 256)])
def test_full_size_synthetic_vs_reference_fingerprints(dq, oracle, golden, tag, kind, w, h, k):
    px = oracle.generate(kind, w, h)
    assert oracle.hash_words(px) == int(golden[f"{tag}_in_hash"][0])
    out, pal = dq.quant_recurse(px, k, 0)
    assert dq.last_stats()["num_points"] == int(golden[f"{tag}_unique"][0])
    assert np.array_equal(pal, golden[f"{tag}_palette"])
    assert oracle.hash_words(out) == int(golden[f"{tag}_out_hash"][0])
    # size-independent properties: every output word is a palette entry; remapping is idempotent;
    # the histogram of the input accounts for every pixel
    assert np.isin(out, pal).all()
    assert np.array_equal(dq.map_colors_mps(out, pal), out)
    col, cnt = dq.histogram(px)
    assert int(cnt.sum()) == px.size and col.size == int(golden[f"{tag}_unique"][0])


def test_split_statistics_within_tolerance(dq, oracle, images):
    px = images["cookie"]
    col, w, cnt = oracle.calc_color_table(px)
    K = 64
    pal, recs, means, sizes = dq.split_points(col, cnt, 1.0 / px.size, K)
    with muted():
        opal, _, orecs = oracle.quant_varpart_fast(px, K, with_records=True)
    assert np.array_equal(pal, opal)
    assert len(orecs) == K - 1
    for g, o in zip(recs, orecs):
        assert (g.new_index, g.old_index, g.cut_axis, g.num_points, g.new_size, g.is_last) == \
               (o.new_index, o.old_index, o.cut_axis, o.num_points, o.new_size, o.is_last)
        scal = [("cut_pos", 1.0), ("total_weight", 0.0), ("new_weight", 0.0), ("old_weight", 0.0)]
        if not o.is_last:
            scal += [("new_tse", 0.0), ("old_tse", 0.0)]
        for f, floor in scal:
            assert abs(getattr(g, f) - getattr(o, f)) <= REL_TOL * max(abs(getattr(o, f)), floor), (o.new_index, f)
        for c in range(3):
            assert abs(g.new_mean[c] - o.new_mean[c]) <= REL_TOL * max(1.0, abs(o.new_mean[c]))
            assert abs(g.old_mean[c] - o.old_mean[c]) <= REL_TOL * max(1.0, abs(o.old_mean[c]))
            if not o.is_last:
                assert abs(g.new_var[c] - o.new_var[c]) <= REL_TOL * max(1.0, abs(o.new_var[c]))
                assert abs(g.old_var[c] - o.old_var[c]) <= REL_TOL * max(1.0, abs(o.old_var[c]))


def test_quant_varpart_parameter_space_vs_model(dq, oracle):
    """num_bits / dec_factor / max_iters / allPixelsUnique.  U <= EXACT_MAX_POINTS: the ordered path, bit-exact against the
    reference semantics; the same inputs with the ordered path switched off exercise the exact-integer kernels,
    bit-exact against the oracle's exact-count model."""
    rng = np.random.default_rng(12)
    c = rng.integers(0, 256, 3)
    n = 40000
    ch = [np.clip(c[j] + rng.integers(-40, 41, n), 0, 255).astype(np.uint32) for j in range(3)]
    px = (ch[0] << 16) | (ch[1] << 8) | ch[2]
    cases = ((16, 8, 1, 10, 0), (16, 6, 1, 10, 0), (64, 5, 2, 3, 0), (300, 8, 1, 10, 0), (9, 7, 3, 1, 1), (32, 8, 1, 5, 1),
             (256, 8, 1, 10, 1))
    assert np.unique(px).size <= EXACT_MAX_POINTS
    for k, bits, dec, iters, uq in cases:
        with muted((2,)):
            pal, empty = dq.quant_varpart_fast(px, k, bits, dec, iters, uq)
        with muted():
            ref, rempty = oracle.quant_varpart_fast(px, k, bits, dec, iters, uq)
        assert np.array_equal(pal, ref) and empty == rempty, (k, bits, dec, iters, uq)
    ctx = dq.lib.dq_default_context()
    dq.lib.dq_context_set_exact_small(ctx, 0)
    try:
        for k, bits, dec, iters, uq in cases:
            with muted((2,)):
                pal, empty = dq.quant_varpart_fast(px, k, bits, dec, iters, uq)
            with muted():
                model, mempty = oracle.quant_varpart_fast(px, k, bits, dec, iters, uq, exact_counts=True)
            assert np.array_equal(pal, model) and empty == mempty, (k, bits, dec, iters, uq)
    finally:
        dq.lib.dq_context_set_exact_small(ctx, 1)


def test_degenerate_inputs(dq, oracle):
    one = np.full(1000, 0x00123456, np.uint32)
    with muted((2,)):
        out, pal = dq.quant_recurse(one, 8, 0)
    with muted():
        oout, opal = oracle.quant_recurse(one, 8, 0)
    assert np.array_equal(pal, opal) and np.array_equal(out, oout) and len(pal) == 1
    # K > U: every pixel maps to itself (SURVEY.md 7)
    rng = np.random.default_rng(3)
    base = rng.integers(0, 1 << 24, 17, dtype=np.uint32)
    px = base[rng.integers(0, 17, 4000)]
    for k in (17, 32, 125, 256, 300):
        with muted((2,)):
            out, pal = dq.quant_recurse(px, k, 0)
        assert len(pal) == 17 and np.array_equal(out, px & 0xFFFFFF), k
    # single pixel
    with muted((2,)):
        out, pal = dq.quant_recurse(np.array([0xFFABCDEF], np.uint32), 4, 0)
    assert list(pal) == [0xABCDEF] and list(out) == [0xABCDEF]


def test_frame_pipeline_matches_single_calls(dq, pkg, oracle):
    import ctypes as C
    import torch
    frames = [oracle.generate(1, 320, 200, 100 + i) for i in range(7)] + [oracle.generate(2, 64, 64, 5)]
    npix = max(f.size for f in frames)
    pipe = pkg.FramePipeline(dq.lib, 0, npix, depth=3)
    ins = [torch.from_numpy(f.view(np.int32).copy()).pin_memory() for f in frames]
    outs = [torch.zeros(f.size, dtype=torch.int32).pin_memory() for f in frames]
    cts = [np.zeros(32, np.uint32) for _ in frames]
    nks = [C.c_uint32(32) for _ in frames]
    for i in range(len(frames)):
        pipe.submit(ins[i].numpy().view(np.uint32), outs[i].numpy().view(np.uint32), 32, cts[i], nks[i], 0)
    ms = pipe.flush()
    assert ms > 0
    for i, f in enumerate(frames):
        with muted((2,)):
            out, pal = dq.quant_recurse(f, 32, 0)
        assert np.array_equal(cts[i][:nks[i].value], pal), i
        assert np.array_equal(outs[i].numpy().view(np.uint32), out), i
    pipe.close()


@pytest.mark.parametrize("lanes,split_ctas", [(1, 0), (4, 0), (8, 9), (5, 148)])
def test_frame_pipeline_lanes_device_frames(dq, pkg, oracle, lanes, split_ctas):
    """Frames in flight on disjoint SM groups: results must not depend on the lane count or the SM partition
    (including an oversubscribed one: 5 lanes that each ask for all SMs simply take turns)."""
    import ctypes as C
    import torch
    shapes = [(320, 200, 1), (64, 64, 2), (500, 333, 1), (17, 3, 2)]
    frames = [oracle.generate(kind, w, h, 200 + i) for i, (w, h, kind) in enumerate(shapes * 4)]
    ks = [(16, 64, 256, 5)[i % 4] for i in range(len(frames))]
    uniq = [1 if i % 5 == 4 else 0 for i in range(len(frames))]
    pipe = pkg.FramePipeline(dq.lib, 0, 0, depth=lanes, split_ctas=split_ctas)
    assert dq.lib.dq_pipeline_lanes(pipe.handle) == lanes
    d_in = [torch.from_numpy(f.view(np.int32).copy()).cuda() for f in frames]
    d_out = [torch.zeros(f.size, dtype=torch.int32, device="cuda") for f in frames]
    cts = [np.zeros(k, np.uint32) for k in ks]
    nks = [C.c_uint32(k) for k in ks]
    torch.cuda.synchronize()
    tickets = [pipe.submit_device(d_in[i].data_ptr(), d_out[i].data_ptr(), frames[i].size, cts[i], nks[i], uniq[i])
               for i in range(len(frames))]
    assert tickets == list(range(len(frames)))
    pipe.wait(tickets[3])     # a single frame can be awaited out of order
    got3 = d_out[3].cpu().numpy().view(np.uint32).copy()
    pipe.flush()
    for i, f in enumerate(frames):
        with muted((2,)):
            out, pal = dq.quant_recurse(f, ks[i], uniq[i])
        assert np.array_equal(cts[i][:nks[i].value], pal), i
        assert np.array_equal(d_out[i].cpu().numpy().view(np.uint32), out), i
        if i == 3:
            assert np.array_equal(got3, out)
    pipe.close()


def test_generic_split_kernel_large_k(dq, oracle, pkg):
    """K > 512 uses the generic split kernel (csrc/dq_split.cu)."""
    rng = np.random.default_rng(21)
    px = rng.integers(0, 1 << 24, 30000, dtype=np.uint32)
    for k in (600, 1000):
        with muted((2,)):
            pal, empty = dq.quant_varpart_fast(px, k, all_unique=1)   # uniform path: bit-exact vs the reference restatement
        with muted():
            opal, oempty = oracle.quant_varpart_fast(px, k, all_unique=1)
        assert np.array_equal(pal, opal) and empty == oempty, k


def test_label_image_matches_oracle(dq, oracle, images, golden):
    # SURVEY.md 8f row 2: mapQuantPixelsToColortableIndexes (OpenCVUtil.cpp:787-849), last duplicate wins
    px = images["cookie"][:200000]
    grid = golden["grid125"]
    quant = dq.map_colors_mps(px, grid)
    assert np.array_equal(dq.colortable_indexes(quant, grid), oracle.colortable_indexes(quant, grid))
    pal = np.array([0x101010, 0x202020, 0x101010, 0x303030, 0xFF202020], np.uint32)
    q = np.array([0x101010, 0x303030, 0x202020, 0x101010], np.uint32)
    assert list(dq.colortable_indexes(q, pal)) == [2, 3, 4, 2]
    assert list(dq.colortable_indexes(q, pal, greyscale=True)) == [0x020202, 0x030303, 0x040404, 0x020202]


def test_ragged_sizes_and_alignment(dq, pkg, oracle):
    """Sizes around the vector widths (4 / 8 pixels per thread), misaligned device pointers, huge palettes."""
    import ctypes as C
    import torch
    rng = np.random.default_rng(33)
    pal = rng.integers(0, 1 << 24, 200, dtype=np.uint32)
    for n in (1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 33, 255, 257, 1023, 1025, 70001):
        px = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
        assert np.array_equal(dq.map_colors_mps(px, pal), oracle.map_colors_mps(px, pal)), n
        col, cnt = dq.histogram(px)
        assert int(cnt.sum()) == n and col.size == np.unique(px & 0xFFFFFF).size, n
    # device pointers that are only 4-byte aligned (row-sharded callers pass offsets into a frame)
    lib = dq.lib
    ctx = lib.dq_default_context()
    base = rng.integers(0, 1 << 24, 500, dtype=np.uint32)
    host = base[rng.integers(0, 500, 100003)]
    dev = torch.from_numpy(host.view(np.int32)).cuda()
    out = torch.zeros_like(dev)
    for off in (1, 2, 3):
        n = host.size - 8
        ct = pal.copy()
        lib.dq_map_colors_device(ctx, dev.data_ptr() + 4 * off, n, out.data_ptr() + 4 * off, ct.ctypes.data_as(C.POINTER(C.c_uint32)),
                                 ct.size, 1)
        assert np.array_equal(out.cpu().numpy().view(np.uint32)[off:off + n], oracle.map_colors_mps(host[off:off + n], pal)), off
        k = C.c_uint32(16)
        ct16 = np.zeros(16, np.uint32)
        lib.dq_quant_recurse_device(ctx, n, dev.data_ptr() + 4 * off, out.data_ptr() + 4 * off, C.byref(k),
                                    ct16.ctypes.data_as(C.POINTER(C.c_uint32)), 0)
        with muted():
            oout, opal = oracle.quant_recurse(host[off:off + n], 16, 0)
        assert np.array_equal(ct16[:k.value], opal) and np.array_equal(out.cpu().numpy().view(np.uint32)[off:off + n], oout), off
    # palette larger than the shared-memory limit of the fast kernels (global-memory fallback)
    big = rng.integers(0, 1 << 24, 9000, dtype=np.uint32)
    px = rng.integers(0, 1 << 24, 3000, dtype=np.uint32)
    assert np.array_equal(dq.map_colors_mps(px, big), oracle.map_colors_mps(px, big))


def test_block_majority_vote(dq, oracle, golden):
    # SURVEY.md 8f row 1: genHistogramsForBlocks (ClusteringSegmentation.cpp:417-563), ties by unordered_map order
    cookie = np.load(_os.path.join(ROOT_DIR, "tests", "golden", "cookie_px.npz"))
    px, (h, w) = cookie["px"].ravel(), cookie["shape"]
    quant, blocks = dq.quant_blocks(px, int(w), int(h), golden["grid125"], 4)   # the live call of the reference pipeline
    assert np.array_equal(quant, oracle.map_colors_mps(px, golden["grid125"]))
    assert np.array_equal(blocks, oracle.block_vote(quant, int(w), int(h), 4))
    # adversarial ties: few colours, every block mixed, ragged borders, all supported block sizes
    rng = np.random.default_rng(9)
    for dim, (ww, hh), ncol in ((4, (203, 101), 3), (4, (64, 64), 40), (2, (33, 17), 2), (3, (50, 31), 5), (8, (95, 70), 70), (1, (9, 5), 4)):
        pal = rng.integers(0, 1 << 24, ncol, dtype=np.uint32)
        q = pal[rng.integers(0, ncol, ww * hh)]
        assert np.array_equal(dq.block_vote(q, ww, hh, dim), oracle.block_vote(q, ww, hh, dim)), (dim, ww, hh, ncol)


def test_pixel_histogram(dq, oracle):
    # SURVEY.md 8f row 2: generatePixelHistogram (OpenCVUtil.cpp:736-781) == np.unique on the 24-bit pixels
    px = oracle.generate(1, 640, 360, 12345)
    keys, counts = dq.pixel_histogram(px)
    ek, ec = np.unique(px & 0xFFFFFF, return_counts=True)
    assert np.array_equal(keys, ek) and np.array_equal(counts, ec)
    keys, counts = dq.pixel_histogram(np.array([0xFF000005, 5, 7], np.uint32))
    assert keys.tolist() == [5, 7] and counts.tolist() == [2, 1]


def test_srm_sorted_edges(dq, oracle, golden):
    """SURVEY.md 8f row 4: SRM's edge list + stable 256-bin sort (SRM/srm.c:135-177, :226-246) -- integer work, bit-exact,
    order inside a bucket included (it is the merge order)."""
    import sys
    sys.path.insert(0, _os.path.join(ROOT_DIR, "tests", "golden"))
    from make_golden import srm_image
    z = np.load(_os.path.join(ROOT_DIR, "tests", "golden", "cookie_px.npz"))
    img = srm_image(z["px"].reshape(int(z["shape"][0]), int(z["shape"][1])))
    pairs = dq.srm_sorted_edges(img)
    assert oracle.hash_words(pairs.reshape(-1)) == int(golden["srm_cookie_pairs_hash"][0])     # the reference's own list
    assert np.array_equal(dq.srm_sorted_edges(np.ascontiguousarray(img[100:137, 200:251])), golden["srm_small_pairs"])
    rng = np.random.default_rng(31)
    for h, w, ch, levels in ((2, 2, 3, 256), (1, 9, 3, 256), (9, 1, 3, 256), (1, 1, 3, 4), (64, 33, 4, 256), (200, 300, 3, 4),
                             (131, 257, 3, 2), (40, 2100, 3, 16), (300, 200, 4, 1)):
        im = (rng.integers(0, levels, (h, w, ch)) * (256 // levels)).astype(np.uint8)
        got, want = dq.srm_sorted_edges(im), oracle.srm_sorted_edges(im)
        assert got.shape == want.shape and np.array_equal(got, want), (h, w, ch, levels)
    assert np.all(np.diff(pairs[:, 2].astype(np.int64)) >= 0)    # sortedness of the full-size list


def test_ordered_path_limits_and_large_k(dq, oracle):
    """K between 1024 and 4096 (per-cluster arrays of the ordered path in global memory, generic split kernel) and the
    run-time limit of the ordered path: below it the reference's result, above it the exact-count model's."""
    rng = np.random.default_rng(41)
    px = rng.integers(0, 1 << 24, 2500, dtype=np.uint32)
    for k in (1025, 1500, 3000):
        with muted():
            ref_out, ref_pal = oracle.quant_recurse(px, k, 0)
        with muted((2,)):
            out, pal = dq.quant_recurse(px, k, 0)
        assert np.array_equal(pal, ref_pal) and np.array_equal(out, ref_out), k
    # K > 512 above the default limit: the generic kernel has no tie audit, so the ordered path takes the input whatever the
    # limit says (19 256 random colours at K = 700 differ from the reference in a palette entry on exact-integer sums)
    px = np.random.default_rng(9).integers(0, 1 << 24, 19300, dtype=np.uint32)
    with muted():
        ref_out, ref_pal = oracle.quant_recurse(px, 700, 0)
    with muted((2,)):
        out, pal = dq.quant_recurse(px, 700, 0)
    assert np.array_equal(pal, ref_pal) and np.array_equal(out, ref_out)
    assert dq.last_stats()["tie_flags"] == 0
    ctx = dq.lib.dq_default_context()
    px = rng.integers(0, 1 << 24, 6000, dtype=np.uint32)
    with muted():
        ref_pal, ref_empty = oracle.quant_varpart_fast(px, 64)
        model, mempty = oracle.quant_varpart_fast(px, 64, exact_counts=True)
    try:
        dq.lib.dq_context_set_exact_max_points(ctx, 10000)   # 6000 colours <= limit: ordered
        with muted((2,)):
            pal, empty = dq.quant_varpart_fast(px, 64)
        assert np.array_equal(pal, ref_pal) and empty == ref_empty
        dq.lib.dq_context_set_exact_max_points(ctx, 5000)    # above the limit: exact-integer kernels ...
        dq.lib.dq_context_set_tie_policy(ctx, 0)             # ... taken at their word (no tie audit)
        with muted((2,)):
            pal, empty = dq.quant_varpart_fast(px, 64)
        assert np.array_equal(pal, model) and empty == mempty
        dq.lib.dq_context_set_tie_policy(ctx, 2)             # default: audited, flagged frames re-run in reference order
        with muted((2,)):
            pal, empty = dq.quant_varpart_fast(px, 64)
        st = dq.last_stats()
        assert np.array_equal(pal, ref_pal) and empty == ref_empty
        assert st["tie_flags"] == 0 or st["ordered_rerun"] == 1 or st["tie_resolved"] > 0 or st["cut_overrides"] > 0
    finally:
        dq.lib.dq_context_set_exact_max_points(ctx, EXACT_DEFAULT_LIMIT)
        dq.lib.dq_context_set_tie_policy(ctx, 2)


def test_ordered_path_above_the_default_limit(dq, oracle, golden):
    """The ordered path goes up to 262 144 colours when asked to: a G1 frame with 68 296 colours on which the exact-integer
    kernels differ from the reference in one palette entry (an exact tie), and the 1080p K=64 BASELINE frame (118 773)."""
    ctx = dq.lib.dq_default_context()
    g1 = oracle.generate(1, 400, 300, 3)
    with muted():
        ref_out, ref_pal = oracle.quant_recurse(g1, 64, 0)
    try:
        dq.lib.dq_context_set_exact_max_points(ctx, 262144)
        with muted((2,)):
            out, pal = dq.quant_recurse(g1, 64, 0)
        assert np.array_equal(pal, ref_pal) and np.array_equal(out, ref_out)
        px = oracle.generate(1, 1920, 1080)
        with muted((2,)):
            out, pal = dq.quant_recurse(px, 64, 0)
        assert np.array_equal(pal, golden["g1_1080_k64_palette"])
        assert oracle.hash_words(out) == int(golden["g1_1080_k64_out_hash"][0])
    finally:
        dq.lib.dq_context_set_exact_max_points(ctx, EXACT_DEFAULT_LIMIT)


def test_frame_pipeline_duplicate_and_equal_sum_palettes(dq, pkg, oracle):
    """The frame pipeline's host palette handling (duplicates dropped, std::sort by r+g+b, lut_init) must equal the
    blocking call frame by frame on the palettes no other pipeline test gives it: duplicate words, many equal r+g+b sums
    (greys), K > U, and K = 300 / 512 (map_unique with uploaded tables)."""
    import ctypes as C
    import torch
    rng = np.random.default_rng(3)
    frames = [oracle.generate(1, 320, 200, 300 + i) for i in range(6)]
    frames.append((rng.integers(0, 256, 5000).astype(np.uint32) * 0x010101))          # greys: every sum distinct by 3
    frames.append(rng.integers(0, 40, 9000).astype(np.uint32) * 0x030201)               # few colours: K > U, duplicates
    frames.append(oracle.generate(2, 96, 96, 9))
    ks = [16, 64, 256, 125, 300, 512, 64, 64, 256]
    pipe = pkg.FramePipeline(dq.lib, 0, 0, depth=4)
    d_in = [torch.from_numpy(f.view(np.int32).copy()).cuda() for f in frames]
    d_out = [torch.zeros(f.size, dtype=torch.int32, device="cuda") for f in frames]
    cts = [np.zeros(k, np.uint32) for k in ks]
    nks = [C.c_uint32(k) for k in ks]
    torch.cuda.synchronize()
    for i in range(len(frames)):
        pipe.submit_device(d_in[i].data_ptr(), d_out[i].data_ptr(), frames[i].size, cts[i], nks[i], 0)
    pipe.flush()
    for i, f in enumerate(frames):
        with muted((2,)):
            out, pal = dq.quant_recurse(f, ks[i], 0)
        assert np.array_equal(cts[i][:nks[i].value], pal), i
        assert np.array_equal(d_out[i].cpu().numpy().view(np.uint32), out), i
    pipe.close()
