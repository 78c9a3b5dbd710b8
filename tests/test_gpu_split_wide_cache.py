"""The split kernel keeps each CTA's shares of a round's wide jobs in shared memory from the cut pass to the partition
(Split2Extra::wide_cache_points, about 12 700 points at K = 256); what does not fit is read from L2 in every pass.  On 9
CTAs (the frame pipeline's default grid at 4K) a CTA's K = 256 share almost fits, on 12 it fits whole, and a CTA with two
or three wide jobs lays their shares out back to back.  Results and the tie audit's verdict must not depend on where the
points come from: checked on these grids against the compiled reference's fingerprints (tests/golden/frames.npz), against
the all-SM grid's verdict, and against the oracle on a Batman crop."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN
from golden import tie_inputs as T
from oracle import muted

pytestmark = pytest.mark.gpu

GRIDS = (9, 12, 0)


@pytest.fixture(scope="module")
def frames():
    return np.load(os.path.join(GOLDEN, "frames.npz"))


def _quantize(dq, ctx, px, k):
    import torch
    d_in = torch.from_numpy(px.view(np.int32).copy()).cuda()
    d_out = torch.empty_like(d_in)
    ct = np.zeros(k, np.uint32)
    nk = C.c_uint32(k)
    torch.cuda.synchronize()
    dq.lib.dq_quant_recurse_device(ctx, px.size, d_in.data_ptr(), d_out.data_ptr(), C.byref(nk), ct.ctypes.data_as(C.POINTER(C.c_uint32)), 0)
    st = dq.last_stats(ctx)
    return ct[:nk.value].copy(), d_out.cpu().numpy().view(np.uint32), st


@pytest.fixture(scope="module")
def grid_ctx(dq):
    ctx = dq.lib.dq_context_create(0)
    yield ctx
    dq.lib.dq_context_destroy(ctx)


GOLDEN_FRAMES = [("c4", s, 64) for s in T.C4_FLAGGED + T.C4_CLEAN[:1]] + \
                [("bench", s, 256) for s in T.BENCH_FLAGGED + (T.BENCH_CLEAN, 12346)]


@pytest.mark.parametrize("tag,seed,k", GOLDEN_FRAMES)
def test_golden_frames_cached_grids(dq, oracle, frames, grid_ctx, tag, seed, k):
    w, h = (1920, 1080) if tag == "c4" else (3840, 2160)
    px = oracle.generate(1, w, h, seed)
    i = int(np.nonzero(frames[f"{tag}_seeds"] == seed)[0][0])
    verdicts = {}
    for g in GRIDS:
        dq.lib.dq_context_set_split_ctas(grid_ctx, g)
        pal, out, st = _quantize(dq, grid_ctx, px, k)
        assert pal.size == int(frames[f"{tag}_pal_size"][i]) and oracle.hash_words(pal) == int(frames[f"{tag}_pal_hash"][i]), (g, "palette")
        assert oracle.hash_words(out) == int(frames[f"{tag}_out_hash"][i]), (g, "output")
        verdicts[g] = (st["tie_flags"], st["tie_resolved"], st["cut_overrides"], st["ordered_rerun"], st["splits_computed"])
    assert len(set(verdicts.values())) == 1, verdicts


def test_batman_crop_cached_grids(dq, oracle, grid_ctx):
    px = np.load(os.path.join(GOLDEN, "batman_px.npz"))["px"].ravel()
    with muted():
        ref_out, ref_pal = oracle.quant_recurse(px, 256, 0)
    for g in GRIDS:
        dq.lib.dq_context_set_split_ctas(grid_ctx, g)
        pal, out, st = _quantize(dq, grid_ctx, px, 256)
        assert np.array_equal(pal, ref_pal), (g, st)
        assert np.array_equal(out, ref_out), (g, st)
