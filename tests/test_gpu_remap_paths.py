"""Every device formulation of map_colors_mps against the oracle, bit for bit, on palettes where most pixels lie at the
same minimal distance from several entries (tests/golden/remap_inputs.py).

The remap picks one of eight formulations from the palette size K, the pointer alignment, the pixel count n and the
number of distinct colours U (csrc/dq_map.cu, csrc/dq_batch.cu); they agree with the reference only if each breaks ties
by the reference's visiting rank.  Each test below forces one formulation, checks from the call's statistics that it
was taken, and compares the output with the oracle:

* brute force (prefer_table = 0): integer arg-min (K <= 512) or float arg-min (<= 8192) with the palette in shared
  memory when the pointers are 16-byte aligned, the keyed loop when they are not, the palette in global memory above
  8192 entries;
* the unique-colour table (prefer_table = 1, n >= 65 536, 4U <= n), with the vector and the scalar gather;
* quant_recurse's remap of its own palette (tables in the kernel's parameter block up to 256 entries);
* the batch remap of many items, each with its own palette, and its label image."""
import ctypes as C

import numpy as np
import pytest

from golden import remap_inputs as R
from oracle import muted

pytestmark = pytest.mark.gpu

KINDS = ("lattice", "star", "grey")
SMEM_LIMIT = 8192                  # map_smem_palette_limit(): larger palettes are read from global memory
SMEM_BYTES = (20, 766 * 4 + 64)    # a shared-memory palette of the float arg-min: 20 bytes per entry + the start table
TABLE_MIN_PIXELS = 1 << 16


def _inputs(oracle, kind, k, n, seed):
    """Tie-dense (pixels, palette, oracle output); the first 512 pixels must keep their ties."""
    px, pal = R.generate(kind, k, n, seed, dup=0.1 if k % 2 else 0.0, alpha=k % 3 == 0)
    if k > 1:
        c = R.tie_classes(px[:512], pal, oracle)
        assert c["multi"] >= 0.2 * 512, (kind, k, c)
    return px, pal, oracle.map_colors_mps(px, pal)


@pytest.fixture(scope="module")
def remap(dq):
    """dq_map_colors_device on the default context, the pixels placed `off` words past a 16-byte boundary."""
    import torch
    lib, ctx = dq.lib, dq.lib.dq_default_context()

    def run(px, pal, prefer_table, off=0):
        n = px.size
        host = np.zeros(n + off + 4, np.uint32)
        host[off:off + n] = px
        dev = torch.from_numpy(host.view(np.int32)).cuda()
        out = torch.zeros_like(dev)
        assert dev.data_ptr() % 16 == 0 and out.data_ptr() % 16 == 0
        ct = np.ascontiguousarray(pal, np.uint32).copy()
        torch.cuda.synchronize()
        lib.dq_map_colors_device(ctx, dev.data_ptr() + 4 * off, n, out.data_ptr() + 4 * off, ct.ctypes.data_as(C.POINTER(C.c_uint32)),
                                 ct.size, prefer_table)
        return out.cpu().numpy().view(np.uint32)[off:off + n].copy(), dq.last_stats()

    return run


@pytest.mark.parametrize("k", R.KS)
@pytest.mark.parametrize("kind", KINDS)
def test_bruteforce(oracle, remap, kind, k):
    """n = 2048 + 0..7 (the 8-pixel blocks and their tail), aligned and 1, 2 or 3 words off."""
    px, pal, want = _inputs(oracle, kind, k, 2048 + 8, seed=7000 + k)
    for off in (0, 1, 2, 3):
        for r in range(8):
            n = 2048 + r
            out, st = remap(px[:n], pal, 0, off)
            assert st["remap_path"] == 1 and st["kernel_launches"] == (2 if k > SMEM_LIMIT else 1), (kind, k, off, n, st)
            bad = np.flatnonzero(out != want[:n])
            assert bad.size == 0, (kind, k, off, n, f"{bad.size} pixels differ, first {int(px[bad[0]]):#x}")


@pytest.mark.parametrize("k", R.KS)
@pytest.mark.parametrize("kind", KINDS)
def test_unique_colour_table(oracle, remap, kind, k):
    """n = 65 536 + 0..7 pixels drawn from at most 8192 colours (4U <= n), aligned (vector gather and its 4-pixel tail)
    and 1 or 3 words off (scalar gather)."""
    pool, pal, pool_want = _inputs(oracle, kind, k, 8192, seed=8000 + k)
    pick = np.random.default_rng(k).integers(0, pool.size, TABLE_MIN_PIXELS + 8)
    px, want = pool[pick], pool_want[pick]
    for off in (0, 1, 3):
        for r in range(8):
            n = TABLE_MIN_PIXELS + r
            out, st = remap(px[:n], pal, 1, off)
            assert st["remap_path"] == 2 and 4 * st["num_points"] <= n, (kind, k, off, n, st)
            # histogram, expand_palette (above the shared-memory limit), map_unique, map_gather, table_clear
            assert st["kernel_launches"] == (5 if k > SMEM_LIMIT else 4), (kind, k, off, n, st)
            bad = np.flatnonzero(out != want[:n])
            assert bad.size == 0, (kind, k, off, n, f"{bad.size} pixels differ, first {int(px[bad[0]]):#x}")


def test_smallest_global_memory_palette_exceeds_shared_memory():
    """K = 11 467 would not fit one block's shared memory as a float arg-min palette, so the table cases at that size
    really need the global-memory palette above map_smem_palette_limit(); 8192 entries do fit."""
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    per_entry, fixed = SMEM_BYTES
    assert per_entry * 11467 + fixed > optin >= per_entry * 11466 + fixed, optin
    assert per_entry * SMEM_LIMIT + fixed <= optin


def test_table_thresholds(oracle, remap):
    """The table path needs n >= 65 536 and 4U <= n: n = 65 535 against 65 536, and U = n/4 against n/4 + 1."""
    rng = np.random.default_rng(5)
    ties, pal = R.generate("lattice", 512, 4096, seed=5)
    ties = np.unique(ties & 0xFFFFFF)
    filler = np.setdiff1d(rng.integers(0, 1 << 24, 40000, dtype=np.uint32), ties)
    for n, u, path in ((65535, 1024, 1), (65536, 1024, 2), (65536, 16384, 2), (65536, 16385, 1)):
        colours = np.concatenate([ties, filler])[:u]
        assert np.unique(colours).size == u
        px = np.concatenate([colours, colours[rng.integers(0, u, n - u)]])[rng.permutation(n)]
        out, st = remap(px, pal, 1)
        assert st["remap_path"] == path, (n, u, st)
        if n >= TABLE_MIN_PIXELS:
            assert st["num_points"] == u, (n, u, st)
        assert np.array_equal(out, oracle.map_colors_mps(px, pal)), (n, u)


@pytest.mark.parametrize("case", R.QUANT_CASES, ids=[f"k{c[0]}" for c in R.QUANT_CASES])
def test_quant_recurse_remap(dq, oracle, case):
    """quant_recurse's remap of the palette it returns, on images whose palettes keep pixels on ties (measured on the
    oracle's palette by tests/test_remap_tie_inputs.py).  The palette itself is compared with the oracle where the
    suite promises it: U <= 65 536 colours and K <= 4096."""
    k, seed, step, colours, reps, _ = case
    px = R.lattice_image(seed, step, colours, reps)
    with muted((2,)):
        out, pal = dq.quant_recurse(px, k, 0)
    st = dq.last_stats()
    assert st["num_points"] == colours
    assert st["remap_path"] == (2 if 2 * colours <= px.size else 1), st
    if k > 11466:
        assert pal.size > 11466
    if k <= 4096:
        with muted():
            _, want_pal = oracle.quant_recurse(px, k, 0)
        assert np.array_equal(pal, want_pal)
    bad = np.flatnonzero(out != oracle.map_colors_mps(px, pal))
    assert bad.size == 0, (k, f"{bad.size} pixels differ, first {int(px[bad[0]]):#x}")


def test_batch_remap(dq, oracle):
    """dq_map_colors_batch on tie-dense items: the palettes of at most 512 entries take the batch kernel, the others the
    single call (one of them with n >= 65 536, 4U <= n and K = 11 467: the table path with a global-memory palette).
    Every item against the oracle, every label against the oracle's colortable_indexes."""
    rng = np.random.default_rng(11)
    items, pals = [], []
    for t in range(90):
        kind = KINDS[t % 3]
        k = R.KS[t % 8] if t % 10 else int(rng.choice([513, 8193]))
        n = 0 if t % 29 == 3 else int(rng.integers(1, 3000))
        px, pal = R.generate(kind, k, n, seed=9000 + t, dup=0.1 if t % 4 == 1 else 0.0, alpha=t % 5 == 2)
        items.append(px)
        pals.append(pal)
    pool, big = R.generate("lattice", 11467, 4096, seed=9999)
    items.append(pool[rng.integers(0, pool.size, TABLE_MIN_PIXELS + 3)])
    pals.append(big)
    res = dq.map_colors_batch(items, pals, labels=True)
    st = dq.last_batch_stats()
    batched = sum(p.size <= 512 for p in pals)
    assert st["items"] == len(items) and st["batched_items"] == batched and st["single_call_items"] == len(items) - batched, st
    assert batched >= 70 and st["single_call_items"] >= 5
    for i, ((out, lab), px, pal) in enumerate(zip(res, items, pals)):
        if px.size == 0:
            continue
        want = oracle.map_colors_mps(px, pal)
        bad = np.flatnonzero(out != want)
        assert bad.size == 0, (i, pal.size, f"{bad.size} pixels differ, first {int(px[bad[0]]):#x}")
        assert np.array_equal(lab, oracle.colortable_indexes(want, pal)), (i, pal.size)
