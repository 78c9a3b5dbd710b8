"""quant_recurse over a batch of small items (dq_quant_recurse_batch_*, csrc/dq_batch.cu).

Every item of a batch must come back exactly as a single quant_recurse call on the same pixels and context returns it:
palette, actual K and output pixels, bit for bit.  A seeded subset is also checked against the oracle."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import muted

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
FUZZ_KS = (1, 2, 3, 4, 5, 16, 64, 125, 256, 300, 512)
EMPTY_LINE = re.compile(r"^# empty clusters: \d+$", re.M)


def _tiles(px, shape, size=32):
    h, w = (int(x) for x in shape)
    img = px.reshape(h, w)
    return [np.ascontiguousarray(img[y:y + size, x:x + size]).ravel() for y in range(0, h, size) for x in range(0, w, size)]


def _fixture(name):
    z = np.load(os.path.join(GOLDEN, f"{name}_px.npz"))
    return z["px"].ravel().astype(np.uint32), z["shape"]


def _fuzz_items(oracle, count, seed):
    """Ragged items of 1 to 20 000 px in the four modes of tools/fuzz_small.py, the colours cut from G1 1080p frames."""
    rng = np.random.default_rng(seed)
    frames = [oracle.generate(1, 1920, 1080, s) for s in (3, 11)]
    items, ks = [], []
    for t in range(count):
        mode = t % 4
        n = int(rng.integers(1, 20001)) if t % 5 else int(rng.integers(1, 300))
        src = frames[t % 2]
        if mode == 0:  # a run of a natural frame
            start = int(rng.integers(0, src.size - n))
            px = src[start:start + n].copy()
        elif mode == 1:  # a few colours of the frame
            pal = src[rng.integers(0, src.size, int(rng.integers(1, 60)))]
            px = pal[rng.integers(0, pal.size, n)]
        elif mode == 2:  # greys: many equal sums
            g = rng.integers(0, 256, int(rng.integers(1, 30)))
            pal = (g * 0x010101).astype(np.uint32)
            px = np.tile(pal, n // pal.size + 1)[:n]
        else:  # 4-level lattice
            c = rng.integers(0, 4, (n, 3)) * 85
            px = ((c[:, 0] << 16) | (c[:, 1] << 8) | c[:, 2]).astype(np.uint32)
        items.append(np.ascontiguousarray(px, np.uint32))
        ks.append(int(rng.choice(FUZZ_KS)))
    # the corner cases: one pixel, one colour, K far above U
    items += [np.array([0x123456], np.uint32), np.full(777, 0x00FF8800, np.uint32), np.array([1, 2, 3, 2, 1], np.uint32)]
    ks += [4, 125, 300]
    return items, ks


def _singles(dq, items, ks, all_unique=0):
    res = []
    for px, k in zip(items, ks):
        res.append(dq.quant_recurse(px, k, all_unique))
    return res


def _assert_same(batch, singles, what=""):
    assert len(batch) == len(singles)
    for i, ((bo, bp), (so, sp)) in enumerate(zip(batch, singles)):
        assert np.array_equal(bp, sp), f"{what} item {i}: palette {bp[:8]} vs {sp[:8]}"
        assert np.array_equal(bo, so), f"{what} item {i}: output pixels differ"


def _batched_by_rule(items, ks, limit=4096, all_unique=0):
    """The selection rule: weighted, K <= 512, at most `limit` distinct colours."""
    return [not all_unique and k <= 512 and np.unique(px & 0xFFFFFF).size <= limit for px, k in zip(items, ks)]


def _check_oracle(oracle, items, ks, batch, count, seed):
    rng = np.random.default_rng(seed)
    for i in rng.choice(len(items), size=min(count, len(items)), replace=False):
        with muted():
            oo, op = oracle.quant_recurse(items[i], ks[i], 0)
        assert np.array_equal(batch[i][1], op), f"item {i}: palette differs from the oracle"
        assert np.array_equal(batch[i][0], oo), f"item {i}: pixels differ from the oracle"


@pytest.mark.parametrize("name", ["cookie", "batman"])
@pytest.mark.parametrize("k", [4, 125])
def test_fixture_tiles_all_batched(dq, oracle, name, k):
    px, shape = _fixture(name)
    items = _tiles(px, shape)
    ks = [k] * len(items)
    with muted((2,)):
        singles = _singles(dq, items, ks)
        batch = dq.quant_recurse_batch(items, ks)
    st = dq.last_batch_stats()
    assert st["items"] == len(items) and st["batched_items"] == len(items) and st["single_call_items"] == 0, st
    _assert_same(batch, singles, f"{name} K={k}")
    _check_oracle(oracle, items, ks, batch, 12, 7)


def test_ragged_fuzz_and_empty_cluster_lines(dq, oracle, capfd):
    items, ks = _fuzz_items(oracle, 500, 2024)
    capfd.readouterr()
    singles = _singles(dq, items, ks)
    single_err = capfd.readouterr().err
    batch = dq.quant_recurse_batch(items, ks)
    batch_err = capfd.readouterr().err
    assert EMPTY_LINE.findall(batch_err) == EMPTY_LINE.findall(single_err)  # the same lines in the same order
    assert len(EMPTY_LINE.findall(batch_err)) > 0
    _assert_same(batch, singles, "fuzz")
    st = dq.last_batch_stats()
    rule = _batched_by_rule(items, ks)
    assert st["batched_items"] == sum(rule) and st["single_call_items"] == len(items) - sum(rule), st
    assert st["batched_items"] > 300
    _check_oracle(oracle, items, ks, batch, 25, 11)


def test_fallback_mix_in_one_batch(dq, oracle, kats):
    items, ks = _fuzz_items(oracle, 120, 77)
    g2 = oracle.generate(2, 1920, 1080, 5).reshape(1080, 1920)
    crops = [np.ascontiguousarray(g2[y:y + 120, x:x + 150]).ravel() for y, x in ((0, 0), (300, 700), (900, 1700))]
    assert all(np.unique(c & 0xFFFFFF).size > 4096 for c in crops)
    items += crops + [items[3], items[8]]
    ks += [64, 256, 125, 600, 700]
    order = np.random.default_rng(1).permutation(len(items))
    items, ks = [items[i] for i in order], [ks[i] for i in order]
    with muted((2,)):
        singles = _singles(dq, items, ks)
        batch = dq.quant_recurse_batch(items, ks)
    _assert_same(batch, singles, "mix")
    st = dq.last_batch_stats()
    rule = _batched_by_rule(items, ks)
    assert st["batched_items"] == sum(rule) and st["single_call_items"] == len(items) - sum(rule), st
    assert st["single_call_items"] >= 5
    # allPixelsUnique = 1: every item takes the single call
    kitems = [np.array(c["pixels"], np.uint32) for c in kats]
    kks = [c["k"] for c in kats]
    with muted((2,)):
        batch = dq.quant_recurse_batch(kitems, kks, all_unique=1)
        singles = _singles(dq, kitems, kks, all_unique=1)
    _assert_same(batch, singles, "kat")
    for c, (out, pal) in zip(kats, batch):
        assert [int(x) for x in pal] == c["palette"] and [int(x) for x in out] == c["out_pixels"], c["name"]
    st = dq.last_batch_stats()
    assert st["batched_items"] == 0 and st["single_call_items"] == len(kats), st


def _ctx_single(lib, ctx, px, k):
    from importlib import import_module
    pkg = import_module("clusteringsegmentation-1_b200")
    px = pkg._u32(px)
    out = np.zeros_like(px)
    ct = np.zeros(max(k, 1), np.uint32)
    nk = C.c_uint32(k)
    lib.dq_quant_recurse_ctx(ctx, px.size, pkg._p(px), pkg._p(out), C.byref(nk), pkg._p(ct), 0)
    return out, ct[:nk.value].copy()


def test_context_settings_move_items_to_the_single_call(dq, oracle):
    items, ks = _fuzz_items(oracle, 80, 5)
    lib = dq.lib
    ctx = lib.dq_context_create(-1)
    try:
        for setting, limit in (("max", 100), ("off", 0)):
            if setting == "max":
                lib.dq_context_set_exact_max_points(ctx, 100)
            else:
                lib.dq_context_set_exact_max_points(ctx, 4096)
                lib.dq_context_set_exact_small(ctx, 0)
            with muted((2,)):
                singles = [_ctx_single(lib, ctx, px, k) for px, k in zip(items, ks)]
                batch = dq.quant_recurse_batch(items, ks, ctx=ctx)
            _assert_same(batch, singles, setting)
            st = dq.last_batch_stats(ctx)
            rule = _batched_by_rule(items, ks, limit) if limit else [False] * len(items)
            assert st["batched_items"] == sum(rule) and st["single_call_items"] == len(items) - sum(rule), (setting, st)
            if limit:
                assert 0 < st["batched_items"] < len(items)
    finally:
        lib.dq_context_destroy(ctx)


def test_items_are_independent(dq, oracle):
    items, ks = _fuzz_items(oracle, 60, 9)
    with muted((2,)):
        whole = dq.quant_recurse_batch(items, ks)
        order = np.random.default_rng(3).permutation(len(items))
        shuffled = dq.quant_recurse_batch([items[i] for i in order], [ks[i] for i in order])
        alone = [dq.quant_recurse_batch([px], [k])[0] for px, k in zip(items, ks)]
    _assert_same([shuffled[j] for j in np.argsort(order)], whole, "shuffled")
    _assert_same(alone, whole, "alone")


def test_device_form_matches_host_form(dq, oracle):
    import torch
    items, ks = _fuzz_items(oracle, 100, 13)
    offsets = np.concatenate([[0], np.cumsum([a.size for a in items])]).astype(np.uint32)
    flat = np.concatenate(items)
    with muted((2,)):
        host = dq.quant_recurse_batch(items, ks)
        d_flat = torch.from_numpy(flat.view(np.int32)).cuda()
        out, pals, nk = dq.quant_recurse_batch_device(d_flat, offsets, ks)
    torch.cuda.synchronize()
    out = out.cpu().numpy().view(np.uint32)
    pal_off = np.concatenate([[0], np.cumsum(ks)])
    for i, (ho, hp) in enumerate(host):
        assert np.array_equal(pals[pal_off[i]:pal_off[i] + nk[i]], hp), i
        assert np.array_equal(out[offsets[i]:offsets[i + 1]], ho), i


def test_launches_do_not_grow_with_items(dq, oracle):
    g1 = oracle.generate(1, 1920, 1080, 21).reshape(1080, 1920)
    tiles = [np.ascontiguousarray(g1[y:y + 24, x:x + 40]).ravel() for y in range(0, 1080, 24) for x in range(0, 1920, 40)]
    launches = []
    for count in (100, 2000):
        with muted((2,)):
            dq.quant_recurse_batch(tiles[:count], [4 if i % 2 else 125 for i in range(count)])
        st = dq.last_batch_stats()
        assert st["batched_items"] == count, st
        assert dq.last_stats()["kernel_launches"] == st["kernel_launches"]
        launches.append(st["kernel_launches"])
    assert launches[0] == launches[1] == 3
