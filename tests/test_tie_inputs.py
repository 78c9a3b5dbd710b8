"""CPU check that the inputs of tests/test_gpu_tie_paths.py (tests/golden/tie_inputs.py) still exercise what they were
chosen for, on the oracle's model of the tie audit and the resolver: the restatement (the reference's arithmetic), the
exact-integer split alone (exact_counts=True) and the integer split with the audit + resolver (quant_varpart_resolved).
If a change of the oracle or of the generator moved an input off its tie, the GPU tests would quietly stop testing the
recovery steps; this file says so without a GPU.  Also the merge rule of the row-sharded path's first-seen indexes."""
import numpy as np
import pytest

from golden import tie_inputs as T
from oracle import muted


def _model(oracle, px, k, bits=8, dec=1, rows=1, cols=None, int_only=True):
    with muted():
        ref, _ = oracle.quant_varpart_fast(px, k, bits, dec, rows=rows, cols=cols)
        res, info = oracle.quant_varpart_resolved(px, k, bits, dec, rows=rows, cols=cols)
        ex = oracle.quant_varpart_fast(px, k, bits, dec, exact_counts=True, rows=rows, cols=cols)[0] if int_only else None
    flagged = info["left"] + info["roundings"] + info["cuts_confirmed"] + info["cuts_forced"]
    return ref, ex, res, info, flagged


def _check_resolved(ref, res, info, flagged, what):
    assert flagged > 0, f"{what}: the audit no longer flags this input"
    assert info["left"] == 0, f"{what}: decisions left for an ordered re-run: {info}"
    assert np.array_equal(res, ref), f"{what}: the resolver model differs from the restatement"


@pytest.mark.parametrize("seed", T.C4_FLAGGED)
def test_c4_flagged_frame_needs_the_resolver(oracle, seed):
    px = oracle.generate(1, 1920, 1080, seed)
    ref, ex, res, info, flagged = _model(oracle, px, 64)
    _check_resolved(ref, res, info, flagged, seed)
    assert (not np.array_equal(ex, ref)) == (seed in T.C4_INT_WRONG), seed
    assert (info["cuts_forced"] >= 1) == (seed == T.C4_FORCED), (seed, info)


@pytest.mark.parametrize("seed", T.C4_CLEAN)
def test_c4_clean_neighbour_is_not_flagged(oracle, seed):
    px = oracle.generate(1, 1920, 1080, seed)
    ref, _, res, info, flagged = _model(oracle, px, 64, int_only=False)
    assert flagged == 0 and np.array_equal(res, ref), (seed, info)


def test_bench_frames_flagged_and_clean(oracle):
    for seed in T.BENCH_FLAGGED + (T.BENCH_CLEAN,):
        px = oracle.generate(1, 3840, 2160, seed)
        ref, _, res, info, flagged = _model(oracle, px, 256, int_only=False)
        if seed == T.BENCH_CLEAN:
            assert flagged == 0 and np.array_equal(res, ref), (seed, info)
        else:
            _check_resolved(ref, res, info, flagged, seed)


@pytest.mark.parametrize("shape", ["1d", "2d"])
def test_varpart_inputs(oracle, shape):
    table = T.VARPART_1D if shape == "1d" else T.VARPART_2D
    rows, cols = (1, None) if shape == "1d" else (1080, 1920)
    assert sum(e[4] for e in table) >= 5 and any(e[5] for e in table)
    for seed, bits, dec, k, int_wrong, forced in table:
        what = (shape, seed, bits, dec, k)
        px = oracle.generate(1, 1920, 1080, seed)
        ref, ex, res, info, flagged = _model(oracle, px, k, bits, dec, rows, cols)
        _check_resolved(ref, res, info, flagged, what)
        assert (not np.array_equal(ex, ref)) == int_wrong, what
        assert (info["cuts_forced"] >= 1) == forced, (what, info)


def test_row_shard_first_seen_merge_rule():
    """dq_rows: every rank exports (colour, shard-local first-seen index) and its pixel count; the merge takes the minimum
    over shards of (sum of the lower shards' pixel counts + local index).  That must be the whole image's first-seen index
    of every colour, whatever the split into row blocks (empty shards included)."""
    rng = np.random.default_rng(7)
    img = rng.integers(0, 300, size=4 * 1000, dtype=np.uint32)  # few colours: many repeat across shards
    uniq, first = np.unique(img, return_index=True)
    for cuts in ([], [2000], [1, 999, 1000, 3999], [0, 0, 4000], sorted(rng.integers(0, 4000, size=7).tolist())):
        bounds = [0] + list(cuts) + [img.size]
        shards = [img[a:b] for a, b in zip(bounds[:-1], bounds[1:])]
        merged = {}
        offset = 0
        for sh in shards:
            u, f = np.unique(sh, return_index=True)
            for c, i in zip(u.tolist(), f.tolist()):
                merged[c] = min(merged.get(c, 1 << 32), offset + i)
            offset += sh.size
        assert sorted(merged) == uniq.tolist(), cuts
        assert [merged[c] for c in uniq.tolist()] == first.tolist(), cuts
