"""map_colors_mps of every region of a tag image, each to its own palette, in one call (dq_map_regions_*,
csrc/dq_regions.cu).

The expected value is always the composition the call replaces, computed here: every region's pixels gathered with numpy
in raster order, dq.map_colors_batch with labels over the mapped regions with pixels, the outputs and labels scattered
back with numpy, a sentinel everywhere else.  Everything must be equal bit for bit."""
import os

import numpy as np
import pytest

from oracle import muted

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
SENTINEL = 0xDEADBEEF


def _fixture(name, oracle):
    if name == "g1":
        return oracle.generate(1, 1920, 1080, 13), 1080, 1920
    z = np.load(os.path.join(GOLDEN, f"{name}_px.npz"))
    h, w = (int(x) for x in z["shape"][:2])
    return z["px"].ravel().astype(np.uint32), h, w


def _voronoi(h, w, cells, seed):
    from scipy.spatial import cKDTree
    pts = np.random.default_rng(seed).random((cells, 2)) * [h, w]
    yy, xx = np.mgrid[0:h, 0:w]
    return cKDTree(pts).query(np.c_[yy.ravel(), xx.ravel()])[1].astype(np.uint32)


def _tile_tags(h, w, size=32):
    yy, xx = np.mgrid[0:h, 0:w]
    return ((yy // size) * (-(-w // size)) + xx // size).ravel().astype(np.uint32)


def _palette(rng, k, frame, t):
    """K entries: colours of a natural frame (mostly absent from the item), lattice colours with many equal sums and
    duplicates, duplicated words, alpha bits."""
    pal = frame[rng.integers(0, frame.size, k)].copy()
    if t % 4 == 1:
        c = rng.integers(0, 4, (k, 3)) * 64
        pal = ((c[:, 0] << 16) | (c[:, 1] << 8) | c[:, 2]).astype(np.uint32)
        pal[::2] = (rng.integers(0, 256, pal[::2].size) * 0x010101).astype(np.uint32)
    if t % 4 == 2:
        pal[rng.integers(0, k, k // 3 + 1)] = pal[rng.integers(0, k)]
    if t % 3 == 0:
        pal |= rng.integers(0, 256, k).astype(np.uint32) << 24
    return np.ascontiguousarray(pal, np.uint32)


def _regions(tags, num):
    """Every region's pixel indexes in raster order."""
    inside = tags < num
    counts = np.bincount(tags[inside], minlength=num)
    order = np.argsort(np.where(inside, tags, num), kind="stable")[:counts.sum()]
    return np.split(order, np.cumsum(counts)[:-1])


def _compose(dq, px, tags, pals):
    """The composition: numpy gather, map_colors_batch with labels over the mapped regions with pixels, numpy scatter.
    Returns (out, labels, idx, items) with SENTINEL at every pixel not written."""
    idx = _regions(tags, len(pals))
    items = [r for r in range(len(pals)) if idx[r].size and pals[r].size]
    res = dq.map_colors_batch([px[idx[r]] for r in items], [pals[r] for r in items], labels=True) if items else []
    out = np.full_like(px, SENTINEL)
    lab = np.full_like(px, SENTINEL)
    for r, (o, l) in zip(items, res):
        out[idx[r]] = o
        lab[idx[r]] = l
    return out, lab, idx, items


def _device(dq, px, tags, pals, labels=True):
    """dq_map_regions_device into buffers that start as SENTINEL; returns numpy (out, labels or None)."""
    import torch
    s = int(np.array([SENTINEL], np.uint32).view(np.int32)[0])
    d_out = torch.full((px.size,), s, dtype=torch.int32, device="cuda")
    d_lab = torch.full((px.size,), s, dtype=torch.int32, device="cuda") if labels else None
    res = dq.map_regions_device(torch.from_numpy(px.view(np.int32)).cuda(), torch.from_numpy(tags.view(np.int32)).cuda(), pals,
                                out=d_out, labels_out=d_lab)
    torch.cuda.synchronize()
    out = (res[0] if labels else res).cpu().numpy().view(np.uint32)
    return out, res[1].cpu().numpy().view(np.uint32) if labels else None


def _host_ctx(dq, pkg, px, tags, pals, labels=True):
    """dq_map_regions_ctx into host buffers that start as SENTINEL: the _ctx form must copy them up."""
    import ctypes as C
    sizes = np.asarray([p.size for p in pals], np.int32)
    ct = np.concatenate([pkg._u32(p) for p in pals] + [np.zeros(1, np.uint32)])
    out = np.full_like(px, SENTINEL)
    lab = np.full_like(px, SENTINEL) if labels else None
    dq.lib.dq_map_regions_ctx(dq.lib.dq_default_context(), px.size, pkg._p(px), pkg._p(tags), len(pals),
                              sizes.ctypes.data_as(C.POINTER(C.c_int)), pkg._p(ct), pkg._p(out), pkg._p(lab) if labels else None)
    return out, lab


def _assert_equal(got, want, what):
    assert np.array_equal(got[0], want[0]), f"{what}: output pixels differ"
    if got[1] is not None:
        assert np.array_equal(got[1], want[1]), f"{what}: labels differ"


def _check_stats(dq, pals, items):
    st = dq.last_batch_stats()
    batched = sum(pals[r].size <= 512 for r in items)
    assert st["items"] == len(pals) and st["empty_clusters"] == 0, st
    assert st["batched_items"] == batched and st["single_call_items"] == len(items) - batched, st
    assert dq.last_stats()["kernel_launches"] == st["kernel_launches"], st


def _check_oracle(oracle, px, pals, idx, items, got, count, seed):
    rng = np.random.default_rng(seed)
    for r in rng.choice(items, size=min(count, len(items)), replace=False):
        oo = oracle.map_colors_mps(px[idx[r]], pals[r])
        assert np.array_equal(got[0][idx[r]], oo), f"region {r}: pixels differ from the oracle"
        assert np.array_equal(got[1][idx[r]], oracle.colortable_indexes(oo, pals[r])), f"region {r}: labels differ from the oracle"


def _quant_palettes(dq, px, tags, num, k):
    """Each region's palette as dq_quant_regions returns it (empty for a region without pixels)."""
    with muted((2,)):
        _, ct, nk = dq.quant_regions(px, tags, [k] * num)
    off = np.concatenate([[0], np.cumsum(np.full(num, k, np.int64))])
    return [ct[off[r]:off[r] + nk[r]].copy() for r in range(num)]


@pytest.mark.parametrize("name", ["cookie", "batman", "g1"])
@pytest.mark.parametrize("layout", ["voronoi", "tiles"])
@pytest.mark.parametrize("palettes", ["grid125", "quant4", "quant125_edited"])
def test_coherent_tags_equal_the_composition(dq, pkg, oracle, golden, name, layout, palettes):
    px, h, w = _fixture(name, oracle)
    tags = _voronoi(h, w, max(4, h * w // 1000), 3) if layout == "voronoi" else _tile_tags(h, w)
    num = int(tags.max()) + 1
    if palettes == "grid125":
        pals = [golden["grid125"].astype(np.uint32)] * num
    elif palettes == "quant4":
        pals = _quant_palettes(dq, px, tags, num, 4)
    else:  # reversed with one entry dropped (the re-sorted palette of :3816, edited as at :2434)
        pals = [p[::-1][:max(1, p.size - 1)].copy() for p in _quant_palettes(dq, px, tags, num, 125)]
    want = _compose(dq, px, tags, pals)
    got = _device(dq, px, tags, pals)
    _assert_equal(got, want, f"{name} {layout} {palettes}")
    _check_stats(dq, pals, want[3])
    if name != "g1":
        _assert_equal(_host_ctx(dq, pkg, px, tags, pals), want, f"{name} {layout} {palettes} (host form)")
    _check_oracle(oracle, px, pals, want[2], want[3], got, 4, 7)


def test_palette_fuzz_with_single_call_regions(dq, oracle):
    # duplicates, alpha bits, equal sums, absent colours; every 23rd palette above 512 entries takes the single call
    px, h, w = _fixture("g1", oracle)
    tags = _voronoi(h, w, 600, 11)
    rng = np.random.default_rng(12)
    frame = oracle.generate(2, 1920, 1080, 4)
    pals = [_palette(rng, int(rng.choice([513, 700, 2000])) if t % 23 == 4 else int(rng.choice([1, 2, 3, 16, 125, 256, 511, 512])),
                     frame, t) for t in range(600)]
    want = _compose(dq, px, tags, pals)
    got = _device(dq, px, tags, pals)
    _assert_equal(got, want, "fuzz")
    _check_stats(dq, pals, want[3])
    st = dq.last_batch_stats()
    assert st["single_call_items"] >= 20 and st["batched_items"] >= 500, st
    _check_oracle(oracle, px, pals, want[2], want[3], got, 12, 3)
    host = dq.map_regions(px, tags, pals, labels=True)
    _assert_equal(host, (np.where(want[0] == SENTINEL, 0, want[0]), np.where(want[1] == SENTINEL, 0, want[1])), "fuzz (host form)")


@pytest.mark.parametrize("regions", [200, 300, 70000, "scattered"])
def test_digit_passes_and_scattered_tags(dq, oracle, regions):
    g1 = oracle.generate(1, 1920, 1080, 23)
    rng = np.random.default_rng(17)
    if regions == 200:
        px, tags = g1[:480 * 270], _voronoi(270, 480, 200, 1)
    elif regions == 300:
        px, tags = g1[:960 * 540], _voronoi(540, 960, 300, 2)
    elif regions == 70000:
        px, tags = g1, (np.arange(g1.size, dtype=np.int64) * 70000 // g1.size).astype(np.uint32)
    else:  # every region spread over the whole crop
        px =np.ascontiguousarray(g1.reshape(1080, 1920)[200:740, 300:1260]).ravel()
        tags = rng.integers(0, 300, px.size).astype(np.uint32)
    num = int(tags.max()) + 1
    pals = [_palette(rng, int(rng.integers(1, 40)) if num > 5000 else int(rng.choice([4, 16, 125, 512])), g1, t) for t in range(num)]
    want = _compose(dq, px, tags, pals)
    got = _device(dq, px, tags, pals)
    _assert_equal(got, want, f"{regions} regions")
    _check_stats(dq, pals, want[3])


def test_unmapped_regions_and_pixels_in_no_region(dq, pkg, oracle, golden):
    px, h, w = _fixture("cookie", oracle)
    tags = _voronoi(h, w, 200, 4)
    tags = np.where(tags % 5 == 0, 1000 + tags, 2 * tags).astype(np.uint32)  # odd regions never occur, some pixels in none
    grid = golden["grid125"].astype(np.uint32)
    rng = np.random.default_rng(2)
    frame = oracle.generate(1, 1920, 1080, 3)
    # empty palettes: regions with pixels (r % 8 == 2) and without (r % 8 == 3); a few palettes above 512 entries
    pals = [np.zeros(0, np.uint32) if r % 8 in (2, 3) else _palette(rng, 600, frame, r) if r % 50 == 4 else grid for r in range(400)]
    want = _compose(dq, px, tags, pals)
    unmapped = np.isin(tags, [r for r in range(400) if r % 8 == 2])
    assert unmapped.any() and (tags >= 400).any()
    for labels in (True, False):
        for form, got in (("device", _device(dq, px, tags, pals, labels)), ("host", _host_ctx(dq, pkg, px, tags, pals, labels))):
            _assert_equal(got, want, f"{form} labels={labels}")
            assert np.all(got[0][unmapped | (tags >= 400)] == SENTINEL)
            _check_stats(dq, pals, want[3])
    # nothing mapped: nothing written
    none = [np.zeros(0, np.uint32)] * 400
    got = _device(dq, px, tags, none)
    assert np.all(got[0] == SENTINEL) and np.all(got[1] == SENTINEL)
    st = dq.last_batch_stats()
    assert st["items"] == 400 and st["batched_items"] == st["single_call_items"] == 0, st


def test_one_region_is_map_colors_mps(dq, oracle, golden):
    px, h, w = _fixture("batman", oracle)
    with muted((2,)):
        _, quant = dq.quant_recurse(px, 125)
    for pal in (golden["grid125"].astype(np.uint32), quant, np.concatenate([quant, np.full(600, 0xFF000000, np.uint32)])):
        out, lab = dq.map_regions(px, np.zeros(px.size, np.uint32), [pal], labels=True)
        single = dq.map_colors_mps(px, pal)
        assert np.array_equal(out, single), pal.size
        assert np.array_equal(lab, dq.colortable_indexes(single, pal)), pal.size
        assert np.array_equal(dq.map_regions(px, np.zeros(px.size, np.uint32), [pal]), single), pal.size


@pytest.mark.parametrize("k", [4, 125])
def test_chain_returns_the_quantized_output_and_labels(dq, oracle, k):
    # map_regions of quant_regions' output with its returned palettes: every output pixel is an entry of its region's
    # deduplicated palette, so output and labels come back unchanged; regions with K = 0 go in as empty palettes
    px, h, w = _fixture("cookie", oracle)
    tags = _voronoi(h, w, 300, 9)
    tags = np.where(tags % 7 == 0, 5000, tags + tags // 10).astype(np.uint32)  # pixels in no region, regions without pixels
    num = int(tags[tags < 5000].max()) + 1
    with muted((2,)):
        qout, ct, nk, qlab = dq.quant_regions(px, tags, [k] * num, labels=True)
    assert (nk == 0).any()
    off = np.concatenate([[0], np.cumsum(np.full(num, k, np.int64))])
    pals = [ct[off[r]:off[r] + nk[r]] for r in range(num)]
    out, lab = dq.map_regions(qout, tags, pals, labels=True)
    assert np.array_equal(out, qout) and np.array_equal(lab, qlab)


def test_device_form_matches_host_form(dq, oracle):
    import torch
    px, h, w = _fixture("g1", oracle)
    tags = _voronoi(h, w, 2000, 6)
    rng = np.random.default_rng(5)
    pals = [np.zeros(0, np.uint32) if t % 97 == 1 else _palette(rng, 900 if t % 101 == 3 else 4 if t % 2 else 125, px, t)
            for t in range(2000)]
    host = dq.map_regions(px, tags, pals, labels=True)
    d_px, d_tags = torch.from_numpy(px.view(np.int32)).cuda(), torch.from_numpy(tags.view(np.int32)).cuda()
    dev = dq.map_regions_device(d_px, d_tags, pals, labels=True)
    plain = dq.map_regions_device(d_px, d_tags, pals)
    torch.cuda.synchronize()
    assert np.array_equal(host[0], dev[0].cpu().numpy().view(np.uint32))
    assert np.array_equal(host[1], dev[1].cpu().numpy().view(np.uint32))
    assert torch.equal(plain, dev[0])
    assert np.array_equal(dq.map_regions(px, tags, pals), host[0])


@pytest.mark.parametrize("cells", [100, 250, 300, 5000])
def test_launches_do_not_grow_with_regions(dq, oracle, cells):
    px = oracle.generate(1, 1920, 1080, 21)[:960 * 540]
    tags = _voronoi(540, 960, cells, 8)
    rng = np.random.default_rng(cells)
    passes = 1 if cells <= 256 else 2
    for unmapped in (False, True):
        pals = [np.zeros(0, np.uint32) if unmapped and r % 9 == 0 else _palette(rng, 4 if r % 2 else 125, px, r) for r in range(cells)]
        for labels in (False, True):
            dq.map_regions(px, tags, pals, labels=labels)
            st = dq.last_batch_stats()
            assert st["single_call_items"] == 0 and st["batched_items"] == sum(
                p.size > 0 and c > 0 for p, c in zip(pals, np.bincount(tags, minlength=cells))), st
            # sort (count, rowscan, scatter per digit pass) + offsets, one batch remap, scatter back
            assert st["kernel_launches"] == 3 * passes + 3, (cells, unmapped, labels, st)
            assert dq.last_stats()["kernel_launches"] == st["kernel_launches"]
