"""map_colors_mps over a batch of items, each with its own palette, with an optional label image
(dq_map_colors_batch_*, csrc/dq_batch.cu).

Every item must come back exactly as a single map_colors_mps call on the same pixels and palette returns it, and its
labels exactly as colortable_indexes of that output in that palette."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
BATCH_KS = (1, 2, 3, 16, 125, 256, 511, 512)
SINGLE_KS = (513, 600, 2000)


def _image(name):
    z = np.load(os.path.join(GOLDEN, f"{name}_px.npz"))
    return z["px"].ravel().astype(np.uint32), tuple(int(x) for x in z["shape"])


def _tiles(px, shape, size=32):
    h, w = shape
    img = px.reshape(h, w)
    return [np.ascontiguousarray(img[y:y + size, x:x + size]).ravel() for y in range(0, h, size) for x in range(0, w, size)]


def _untile(tiles, shape, size=32):
    h, w = shape
    img = np.zeros((h, w), np.uint32)
    it = iter(tiles)
    for y in range(0, h, size):
        for x in range(0, w, size):
            t = next(it)
            th, tw = min(size, h - y), min(size, w - x)
            img[y:y + th, x:x + tw] = t.reshape(th, tw)
    return img.ravel()


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


def _fuzz(oracle, count, seed):
    """Ragged items of 0 to 20 000 px (some empty) with palettes of the batched sizes and a few above 512."""
    rng = np.random.default_rng(seed)
    frame = oracle.generate(1, 1920, 1080, 3)
    items, pals = [], []
    for t in range(count):
        n = 0 if t % 41 == 5 else int(rng.integers(1, 20001)) if t % 5 else int(rng.integers(1, 300))
        if t % 3 == 0:  # a run of a natural frame
            start = int(rng.integers(0, frame.size - n))
            px = frame[start:start + n].copy()
        elif t % 3 == 1:  # greys and a coarse lattice: ties in the sums and in the distances
            c = rng.integers(0, 5, (n, 3)) * 63
            px = ((c[:, 0] << 16) | (c[:, 1] << 8) | c[:, 2]).astype(np.uint32)
            px[::2] = (rng.integers(0, 256, px[::2].size) * 0x010101).astype(np.uint32)
        else:  # anything, alpha included
            px = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
        k = int(rng.choice(SINGLE_KS)) if t % 23 == 4 else int(rng.choice(BATCH_KS))
        items.append(np.ascontiguousarray(px, np.uint32))
        pals.append(_palette(rng, k, frame, t))
    return items, pals


@pytest.fixture(scope="module")
def fuzz(oracle):
    return _fuzz(oracle, 500, 2025)


@pytest.fixture(scope="module")
def fuzz_singles(dq, fuzz):
    items, pals = fuzz
    return [dq.map_colors_mps(px, p) if px.size else px.copy() for px, p in zip(items, pals)]


def _assert_outputs(batch, singles, what=""):
    assert len(batch) == len(singles)
    for i, (b, s) in enumerate(zip(batch, singles)):
        assert np.array_equal(b, s), f"{what} item {i}: output pixels differ"


@pytest.mark.parametrize("name", ["cookie", "batman"])
def test_fixture_tiles_to_grid125(dq, golden, oracle, name):
    px, shape = _image(name)
    grid = golden["grid125"]
    items = _tiles(px, shape)
    batch = dq.map_colors_batch(items, [grid] * len(items))
    st = dq.last_batch_stats()
    assert st["items"] == len(items) and st["batched_items"] == len(items) and st["single_call_items"] == 0, st
    _assert_outputs(batch, [dq.map_colors_mps(t, grid) for t in items], name)
    assert oracle.hash_words(_untile(batch, shape)) == int(golden[f"{name}_grid125_out_hash"][0])  # the reference's output


@pytest.mark.parametrize("k", [4, 125])
def test_tiles_to_their_own_quantized_palettes(dq, k):
    from oracle import muted
    px, shape = _image("cookie")
    items = _tiles(px, shape)
    with muted((2,)):
        quant = dq.quant_recurse_batch(items, [k] * len(items))
    pals = [p for _, p in quant]
    batch = dq.map_colors_batch(items, pals)
    assert dq.last_batch_stats()["batched_items"] == len(items)
    _assert_outputs(batch, [dq.map_colors_mps(t, p) for t, p in zip(items, pals)], f"K={k}")
    _assert_outputs(batch, [o for o, _ in quant], f"K={k} vs the quant batch")


def test_ragged_fuzz(dq, oracle, fuzz, fuzz_singles):
    items, pals = fuzz
    batch = dq.map_colors_batch(items, pals)
    _assert_outputs(batch, fuzz_singles, "fuzz")
    st = dq.last_batch_stats()
    batched = sum(p.size <= 512 for p in pals)
    assert st["items"] == len(items) and st["empty_clusters"] == 0, st
    assert st["batched_items"] == batched and st["single_call_items"] == len(items) - batched, st
    assert 0 < st["single_call_items"] < 50 and any(px.size == 0 for px in items)
    rng = np.random.default_rng(8)
    for i in rng.choice(len(items), 30, replace=False):
        assert np.array_equal(batch[i], oracle.map_colors_mps(items[i], pals[i])), f"item {i}: differs from the oracle"


def test_labels(dq, fuzz, fuzz_singles):
    items, pals = fuzz
    batch = dq.map_colors_batch(items, pals, labels=True)
    assert dq.last_batch_stats()["single_call_items"] > 0
    _assert_outputs([o for o, _ in batch], fuzz_singles, "with labels")
    for i, ((out, lab), p) in enumerate(zip(batch, pals)):
        assert np.array_equal(lab, dq.colortable_indexes(out, p)), f"item {i} (K={p.size}): labels differ"
    # the last duplicate wins, whatever its alpha byte; a palette above 512 entries takes the single call
    pal = np.array([0x102030, 0x405060, 0xFF102030, 0x708090, 0x405060, 0x00102030 | 0x7F000000], np.uint32)
    px = np.array([0x102030, 0x111F31, 0x405060, 0xAA708090, 0x7F8F9F], np.uint32)
    big = np.concatenate([pal, np.full(600, 0x00FFFFFF, np.uint32), [0x405060]]).astype(np.uint32)
    (o1, l1), (o2, l2) = dq.map_colors_batch([px, px], [pal, big], labels=True)
    assert [int(x) for x in o1] == [0x102030, 0x102030, 0x405060, 0x708090, 0x708090]
    assert [int(x) for x in l1] == [5, 5, 4, 3, 3]
    assert np.array_equal(o2, o1) and [int(x) for x in l2] == [5, 5, 606, 3, 3]


def test_items_are_independent(dq, fuzz):
    items, pals = (x[:80] for x in fuzz)
    whole = dq.map_colors_batch(items, pals, labels=True)
    order = np.random.default_rng(4).permutation(len(items))
    shuffled = dq.map_colors_batch([items[i] for i in order], [pals[i] for i in order], labels=True)
    alone = [dq.map_colors_batch([px], [p], labels=True)[0] for px, p in zip(items, pals)]
    for j, i in enumerate(order):
        assert np.array_equal(shuffled[j][0], whole[i][0]) and np.array_equal(shuffled[j][1], whole[i][1]), i
    for i, (a, w) in enumerate(zip(alone, whole)):
        assert np.array_equal(a[0], w[0]) and np.array_equal(a[1], w[1]), i


def test_device_form_matches_host_form(dq, fuzz):
    import torch
    items, pals = (x[:150] for x in fuzz)
    offsets = np.concatenate([[0], np.cumsum([a.size for a in items])]).astype(np.uint32)
    host = dq.map_colors_batch(items, pals, labels=True)
    d_flat = torch.from_numpy(np.concatenate(items).view(np.int32)).cuda()
    out, lab = dq.map_colors_batch_device(d_flat, offsets, pals, labels=True)
    out_nl, lab_nl = dq.map_colors_batch_device(d_flat, offsets, pals)
    torch.cuda.synchronize()
    assert lab_nl is None and torch.equal(out, out_nl)
    out, lab = out.cpu().numpy().view(np.uint32), lab.cpu().numpy().view(np.uint32)
    for i, (ho, hl) in enumerate(host):
        assert np.array_equal(out[offsets[i]:offsets[i + 1]], ho), i
        assert np.array_equal(lab[offsets[i]:offsets[i + 1]], hl), i


def test_one_launch_when_all_items_are_batched(dq, oracle):
    g1 = oracle.generate(1, 1920, 1080, 21).reshape(1080, 1920)
    tiles = [np.ascontiguousarray(g1[y:y + 24, x:x + 40]).ravel() for y in range(0, 1080, 24) for x in range(0, 1920, 40)]
    rng = np.random.default_rng(6)
    pals = [g1.ravel()[rng.integers(0, g1.size, 4 if i % 2 else 125)] for i in range(len(tiles))]
    for count in (100, 2000):
        for labels in (False, True):
            dq.map_colors_batch(tiles[:count], pals[:count], labels=labels)
            st = dq.last_batch_stats()
            assert st["batched_items"] == count and st["kernel_launches"] == 1, (count, labels, st)
            assert dq.last_stats()["kernel_launches"] == 1
