"""The split kernel's results do not depend on its grid, where its CTAs take different shares of the work: on 1 CTA every
job is local, on 4 and 8 (the frame pipeline's lanes) a CTA takes part in several wide jobs per pass and a wide job spans
several CTAs, and each of those jobs stops at the 2-means fixed point on its own; narrow jobs of up to 2048 points run two
at a time in 8-warp groups of a CTA, larger ones on the whole CTA; 0 = as many CTAs as fit on the device.
Checked against the compiled reference's fingerprints (tests/golden/frames.npz) on the golden frames the tie audit flags
and on clean ones, with the audit's verdict (tie_flags / tie_resolved / cut_overrides) the same on every grid, and against
the oracle at K = 3, K = 512 and on a Batman crop."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN
from golden import tie_inputs as T
from oracle import muted

pytestmark = pytest.mark.gpu

GRIDS = (1, 4, 8, 0)


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
def test_golden_frames_every_grid(dq, oracle, frames, grid_ctx, tag, seed, k):
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
    if frames[f"{tag}_tie_mask"][i] != 0:
        assert verdicts[0][0] != 0, verdicts


@pytest.mark.parametrize("k", [3, 512])
def test_bench_frame_k_every_grid(dq, oracle, grid_ctx, k):
    px = oracle.generate(1, 3840, 2160, T.BENCH_CLEAN)
    with muted():
        ref_out, ref_pal = oracle.quant_recurse(px, k, 0)
    for g in GRIDS:
        dq.lib.dq_context_set_split_ctas(grid_ctx, g)
        pal, out, st = _quantize(dq, grid_ctx, px, k)
        assert np.array_equal(pal, ref_pal), (g, k, st)
        assert np.array_equal(out, ref_out), (g, k, st)


def test_batman_crop_every_grid(dq, oracle, grid_ctx):
    px = np.load(os.path.join(GOLDEN, "batman_px.npz"))["px"].ravel()
    with muted():
        ref_out, ref_pal = oracle.quant_recurse(px, 256, 0)
    for g in GRIDS:
        dq.lib.dq_context_set_split_ctas(grid_ctx, g)
        pal, out, st = _quantize(dq, grid_ctx, px, 256)
        assert np.array_equal(pal, ref_pal), (g, st)
        assert np.array_equal(out, ref_out), (g, st)
