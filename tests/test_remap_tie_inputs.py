"""CPU check of the remap's tie inputs (tests/golden/remap_inputs.py) and of the claim every device remap rests on.

On palettes where most pixels lie at the same minimal distance from several entries, the oracle's pruned walk (the
reference's map_colors_mps restated), its (dist, rank) brute force and the plain numpy argmin of remap_inputs must all
agree, at every palette size around the device's switches; so must the compiled reference where it is present.  Every
input must also keep its share of tie pixels: tests/test_gpu_remap_paths.py runs the same generators on the device, and
an input that drifted off its ties would let a wrong tie-break pass there."""
import numpy as np
import pytest

from golden import remap_inputs as R
from oracle import muted

# numpy reference bound: K * n int64 distances per input
WORK = 1 << 24
KINDS = ("lattice", "star", "grey")


def _case(kind, k):
    n = max(64, min(3000, WORK // k))
    # duplicate words for odd K, alpha bytes for K divisible by 3, both now and then
    return R.generate(kind, k, n, seed=1000 * KINDS.index(kind) + k, dup=0.1 if k % 2 else 0.0, alpha=k % 3 == 0)


def _floor(kind, k, n, c):
    """The share of tie pixels each kind keeps (measured: lattice 27-97 % multi, star 46-100 %, grey 44-87 %)."""
    if k == 1:
        assert c["multi"] == 0
        return
    assert c["multi"] >= 0.3 * n, (kind, k, c)
    if kind == "lattice":
        assert c["inside"] >= 0.2 * n, (kind, k, c)
    if kind == "star" and k > 3:
        assert c["inside"] >= 0.3 * n, (kind, k, c)
    if kind == "grey" and k > 3:
        assert c["below"] >= 0.1 * n and c["above"] >= 0.1 * n, (kind, k, c)


@pytest.mark.parametrize("k", R.KS)
@pytest.mark.parametrize("kind", KINDS)
def test_walk_bruteforce_and_numpy_agree(oracle, kind, k):
    px, pal = _case(kind, k)
    assert pal.size == k
    walk = oracle.map_colors_mps(px, pal)
    assert np.array_equal(walk, oracle.map_colors_mps(px, pal, bruteforce=True)), (kind, k)
    assert np.array_equal(walk, R.nearest_dist_rank(px, pal, oracle)), (kind, k)
    _floor(kind, k, px.size, R.tie_classes(px, pal, oracle))


def test_tie_classes_cover_every_start_position(oracle):
    """Across the inputs the start index lies inside the run of equidistant entries, below it and above it: the three
    branches of the integer resolver and both walking directions of the float one."""
    total = {"inside": 0, "below": 0, "above": 0}
    for kind in KINDS:
        for k in (3, 257, 8193):
            c = R.tie_classes(*_case(kind, k), oracle)
            for key in total:
                total[key] += c[key]
    assert min(total.values()) >= 500, total


@pytest.mark.parametrize("kind", KINDS)
def test_compiled_reference_agrees(reference, oracle, kind):
    for k in R.KS:
        px, pal = _case(kind, k)
        assert np.array_equal(reference.map_colors_mps(px, pal), oracle.map_colors_mps(px, pal)), (kind, k)


def test_numpy_reference_by_hand(oracle):
    """nearest_dist_rank on a case worked out by hand: (16, 0, 0) is 16 away from (0, 0, 0) and (32, 0, 0); sorted by
    sum the palette is [0x000000, 0x200000, 0x400000], the start index of sum 16 is 1 (the midpoint of 0 and 32 rounds
    up), so rank 0 goes to 0x200000."""
    pal = np.array([0x400000, 0x000000, 0x200000], np.uint32)
    px = np.array([0x100000, 0x300000, 0x00000F], np.uint32)
    want = [0x200000, 0x400000, 0x000000]
    assert R.nearest_dist_rank(px, pal, oracle).tolist() == want
    assert oracle.map_colors_mps(px, pal).tolist() == want
    assert R.tie_classes(px, pal, oracle) == {"multi": 2, "inside": 2, "below": 0, "above": 0}


@pytest.mark.parametrize("case", R.QUANT_CASES, ids=[f"k{c[0]}" for c in R.QUANT_CASES])
def test_quant_inputs_put_pixels_on_ties(oracle, case):
    """The quant_recurse inputs of the GPU test: the oracle's palette for them keeps pixels on ties (random images put
    0-0.25 % there), with 2U <= n except for the last, and above 11 466 entries for K = 12 000."""
    k, seed, step, colours, reps, share = case
    px = R.lattice_image(seed, step, colours, reps)
    with muted():
        out, pal = oracle.quant_recurse(px, k, 0)
    assert (2 * colours <= px.size) == (reps > 1)
    if k > 11466:
        assert pal.size > 11466
    sub = px[:max(2000, WORK // pal.size)]
    c = R.tie_classes(sub, pal, oracle)
    assert c["multi"] >= share * sub.size, (k, c)
    assert np.array_equal(out[:sub.size], R.nearest_dist_rank(sub, pal, oracle))
