"""quant_recurse of every region of a tag image in one call (dq_quant_regions_*, csrc/dq_regions.cu).

The expected value is always the composition the call replaces, computed here: every region's pixels gathered with numpy
in raster order, dq.quant_recurse_batch over the regions with pixels, the outputs scattered back with numpy, the labels
from dq.colortable_indexes.  Everything must be equal bit for bit."""
import os
import re

import numpy as np
import pytest

from oracle import muted

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
EMPTY_LINE = re.compile(r"^# empty clusters: \d+$", re.M)
SENTINEL = 0xDEADBEEF


def _fixture(name):
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


def _compose(dq, px, tags, ks, labels=True, label_regions=None):
    """The composition: numpy gather, quant_recurse_batch, numpy scatter, colortable_indexes per region.  Returns
    (out, {region: palette}, actual K, labels) with 0 at pixels in no region; labels only for label_regions (all when
    None)."""
    num = len(ks)
    inside = tags < num
    counts = np.bincount(tags[inside], minlength=num)
    order = np.argsort(np.where(inside, tags, num), kind="stable")[:counts.sum()]
    idx = np.split(order, np.cumsum(counts)[:-1])
    nonempty = [r for r in range(num) if counts[r]]
    res = dq.quant_recurse_batch([px[idx[r]] for r in nonempty], [ks[r] for r in nonempty]) if nonempty else []
    out, lab = np.zeros_like(px), np.zeros_like(px)
    pals, nk = {}, np.zeros(num, np.uint32)
    for r, (o, p) in zip(nonempty, res):
        out[idx[r]] = o
        pals[r] = p
        nk[r] = p.size
        if labels and (label_regions is None or r in label_regions):
            lab[idx[r]] = dq.colortable_indexes(o, p)
    return out, pals, nk, lab, idx


def _assert_regions(got, want, ks, what, label_regions=None):
    out, ct, nk = got[:3]
    wout, wpals, wnk, wlab, idx = want
    assert np.array_equal(nk, wnk), f"{what}: actual K differs"
    pal_off = np.concatenate([[0], np.cumsum(np.asarray(ks, np.int64))])
    for r, p in wpals.items():
        assert np.array_equal(ct[pal_off[r]:pal_off[r] + nk[r]], p), f"{what} region {r}: palette differs"
    assert np.array_equal(out, wout), f"{what}: output pixels differ"
    if len(got) > 3:
        if label_regions is None:
            assert np.array_equal(got[3], wlab), f"{what}: labels differ"
        else:
            for r in label_regions:
                assert np.array_equal(got[3][idx[r]], wlab[idx[r]]), f"{what} region {r}: labels differ"


def _check_oracle(oracle, px, idx, ks, got, count, seed):
    out, ct, nk = got[:3]
    pal_off = np.concatenate([[0], np.cumsum(np.asarray(ks, np.int64))])
    rng = np.random.default_rng(seed)
    regions = [r for r in range(len(ks)) if idx[r].size]
    for r in rng.choice(regions, size=min(count, len(regions)), replace=False):
        with muted():
            oo, op = oracle.quant_recurse(px[idx[r]], ks[r], 0)
        assert np.array_equal(ct[pal_off[r]:pal_off[r] + nk[r]], op), f"region {r}: palette differs from the oracle"
        assert np.array_equal(out[idx[r]], oo), f"region {r}: pixels differ from the oracle"


@pytest.mark.parametrize("name", ["cookie", "batman"])
@pytest.mark.parametrize("layout", ["voronoi", "tiles"])
@pytest.mark.parametrize("k", [4, 125])
def test_coherent_tags_equal_the_composition(dq, oracle, name, layout, k):
    px, h, w = _fixture(name)
    tags = _voronoi(h, w, max(4, h * w // 1000), 3) if layout == "voronoi" else _tile_tags(h, w)
    ks = [k] * (int(tags.max()) + 1)
    with muted((2,)):
        want = _compose(dq, px, tags, ks)
        got = dq.quant_regions(px, tags, ks, labels=True)
    _assert_regions(got, want, ks, f"{name} {layout} K={k}")
    st = dq.last_batch_stats()
    assert st["items"] == len(ks) and st["batched_items"] + st["single_call_items"] == sum(i.size > 0 for i in want[4]), st
    _check_oracle(oracle, px, want[4], ks, got, 4, 7)


def test_scattered_random_tags(dq, oracle):
    # every region is spread over the whole crop: an unstable partition would change the first-seen order of its colours
    g1 = oracle.generate(1, 1920, 1080, 17).reshape(1080, 1920)
    px = np.ascontiguousarray(g1[200:740, 300:1260]).ravel()
    tags = np.random.default_rng(5).integers(0, 300, px.size).astype(np.uint32)
    ks = [16 if r % 3 else 64 for r in range(300)]
    with muted((2,)):
        want = _compose(dq, px, tags, ks)
        got = dq.quant_regions(px, tags, ks, labels=True)
    _assert_regions(got, want, ks, "scattered")
    _check_oracle(oracle, px, want[4], ks, got, 3, 9)


@pytest.mark.parametrize("regions", ["one_pass", "two_passes", "three_passes"])
def test_digit_passes(dq, oracle, regions):
    g1 = oracle.generate(1, 1920, 1080, 23)
    if regions == "one_pass":
        px, tags = g1[:480 * 270], _voronoi(270, 480, 256, 1)
        ks = [4 if r % 2 else 125 for r in range(256)]
    elif regions == "two_passes":
        px, tags = g1, _voronoi(1080, 1920, 5000, 2)
        ks = [4 if r % 2 else 32 for r in range(5000)]
    else:
        px, tags = g1, (np.arange(g1.size) // 16).astype(np.uint32)
        ks = [4] * int(tags.max() + 1)
        assert len(ks) > 65536
    label_regions = None if len(ks) <= 5000 else set(range(0, len(ks), 997))
    with muted((2,)):
        want = _compose(dq, px, tags, ks, label_regions=label_regions)
        got = dq.quant_regions(px, tags, ks, labels=True)
    _assert_regions(got, want, ks, regions, label_regions)
    assert dq.last_batch_stats()["items"] == len(ks)


def test_single_call_mix_and_empty_cluster_lines(dq, oracle, capfd):
    g2 = oracle.generate(2, 1920, 1080, 5).reshape(1080, 1920)
    px = np.ascontiguousarray(g2[300:780, 600:1240]).ravel()  # 480 x 640
    tags = _tile_tags(480, 640, 160)  # 12 regions of 25 600 px, most above 4096 colours
    g1 = oracle.generate(1, 1920, 1080, 11)
    px = np.concatenate([px, g1[:200 * 640]])  # and 40 small regions of G1 below the 4096-colour limit
    tags = np.concatenate([tags, 12 + (np.arange(200 * 640) // 3200).astype(np.uint32)])
    ks = [64, 256, 600, 125, 4, 700, 16, 600, 300, 8, 2, 512] + [600 if r % 7 == 0 else 1 + r % 40 for r in range(40)]
    capfd.readouterr()
    want = _compose(dq, px, tags, ks, labels=False)
    want_err = capfd.readouterr().err
    got = dq.quant_regions(px, tags, ks)
    got_err = capfd.readouterr().err
    assert EMPTY_LINE.findall(got_err) == EMPTY_LINE.findall(want_err)
    _assert_regions(got, want, ks, "mix")
    items = [px[i] for i in want[4]]
    rule = [k <= 512 and np.unique(p & 0xFFFFFF).size <= 4096 for p, k in zip(items, ks)]
    st = dq.last_batch_stats()
    assert st["batched_items"] == sum(rule) and st["single_call_items"] == len(ks) - sum(rule), st
    assert st["single_call_items"] >= 9 and st["batched_items"] >= 20, st


def test_empty_regions_and_pixels_in_no_region(dq, oracle):
    import torch
    px, h, w = _fixture("cookie")
    tags = _voronoi(h, w, 200, 4)
    tags = np.where(tags % 5 == 0, 1000 + tags, 2 * tags).astype(np.uint32)  # odd regions never occur, some pixels in none
    ks = [8 + r % 50 for r in range(400)]
    with muted((2,)):
        want = _compose(dq, px, tags, ks)
        sentinel = int(np.array([SENTINEL], np.uint32).view(np.int32)[0])
        d_out = torch.full((px.size,), sentinel, dtype=torch.int32, device="cuda")
        d_lab = torch.full((px.size,), sentinel, dtype=torch.int32, device="cuda")
        out, ct, nk, lab = dq.quant_regions_device(torch.from_numpy(px.view(np.int32)).cuda(), torch.from_numpy(tags.view(np.int32)).cuda(),
                                                   ks, out=d_out, labels_out=d_lab)
    out, lab = out.cpu().numpy().view(np.uint32), lab.cpu().numpy().view(np.uint32)
    inside = tags < len(ks)
    assert (~inside).any() and np.all(out[~inside] == SENTINEL) and np.all(lab[~inside] == SENTINEL)
    _assert_regions((np.where(inside, out, 0), ct, nk, np.where(inside, lab, 0)), want, ks, "empty regions")
    pal_off = np.concatenate([[0], np.cumsum(ks)])
    for r in range(1, len(ks), 2):
        assert nk[r] == 0 and not ct[pal_off[r]:pal_off[r + 1]].any(), r
    st = dq.last_batch_stats()
    assert st["items"] == len(ks) and st["batched_items"] + st["single_call_items"] == sum(i.size > 0 for i in want[4]), st


def test_one_region_is_quant_recurse(dq, oracle):
    px, h, w = _fixture("batman")
    for k in (4, 125):
        with muted((2,)):
            out, ct, nk, lab = dq.quant_regions(px, np.zeros(px.size, np.uint32), [k], labels=True)
            sout, spal = dq.quant_recurse(px, k)
        assert np.array_equal(ct[:nk[0]], spal) and np.array_equal(out, sout), k
        assert np.array_equal(lab, dq.colortable_indexes(sout, spal)), k


def test_device_form_matches_host_form(dq, oracle):
    import torch
    g1 = oracle.generate(1, 1920, 1080, 31)
    tags = _voronoi(1080, 1920, 2000, 6)
    ks = [4 if r % 2 else 125 for r in range(2000)]
    with muted((2,)):
        host = dq.quant_regions(g1, tags, ks, labels=True)
        d_px, d_tags = torch.from_numpy(g1.view(np.int32)).cuda(), torch.from_numpy(tags.view(np.int32)).cuda()
        dev = dq.quant_regions_device(d_px, d_tags, ks, labels=True)
        plain = dq.quant_regions_device(d_px, d_tags, ks)
    torch.cuda.synchronize()
    for a, b in zip(host, dev):
        assert np.array_equal(a, b.cpu().numpy().view(np.uint32) if torch.is_tensor(b) else b)
    assert np.array_equal(plain[0].cpu().numpy(), dev[0].cpu().numpy()) and np.array_equal(plain[1], dev[1])


def test_launches_do_not_grow_with_regions(dq, oracle):
    px = oracle.generate(1, 1920, 1080, 21)[:480 * 270]
    launches = []
    for cells in (100, 250):
        tags = _voronoi(270, 480, cells, 8)
        with muted((2,)):
            dq.quant_regions(px, tags, [4 if r % 2 else 125 for r in range(cells)], labels=True)
        st = dq.last_batch_stats()
        assert st["batched_items"] == st["items"] - (np.bincount(tags, minlength=cells) == 0).sum(), st
        assert st["single_call_items"] == 0 and dq.last_stats()["kernel_launches"] == st["kernel_launches"], st
        launches.append(st["kernel_launches"])
    # sort (count, rowscan, scatter) + offsets, batch histogram + split + remap, scatter back
    assert launches[0] == launches[1] == 4 + 3 + 1
