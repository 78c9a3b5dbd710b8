"""The tie audit's recovery steps (resolver, forced cut, ordered re-run) on every entry path that has its own control flow
around them, against the reference: fingerprints of the compiled reference (tests/golden/frames.npz) for the golden frames,
the oracle's restatement (pinned bit-identical to the reference by test_oracle_golden.py) for quant_varpart_fast with
num_bits < 8 / dec_factor > 1.  The inputs are chosen on the CPU model (tests/golden/tie_inputs.py; test_tie_inputs.py
checks they still hit their ties).  test_gpu_frames.py covers the blocking quant_recurse on the default context."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from golden import tie_inputs as T
from oracle import muted

pytestmark = pytest.mark.gpu

C4 = ("c4", 1920, 1080, 64)
BENCH = ("bench", 3840, 2160, 256)


@pytest.fixture(scope="module")
def frames():
    return np.load(os.path.join(GOLDEN, "frames.npz"))


@pytest.fixture(scope="module")
def images(oracle):
    """(tag, seed) -> pixels of the golden frames used here."""
    out = {}
    for seed in T.C4_FLAGGED + T.C4_CLEAN:
        out[("c4", seed)] = oracle.generate(1, 1920, 1080, seed)
    for seed in T.BENCH_FLAGGED + (T.BENCH_CLEAN,):
        out[("bench", seed)] = oracle.generate(1, 3840, 2160, seed)
    return out


def _golden(frames, tag, seed):
    i = int(np.nonzero(frames[f"{tag}_seeds"] == seed)[0][0])
    return (int(frames[f"{tag}_pal_size"][i]), int(frames[f"{tag}_pal_hash"][i]), int(frames[f"{tag}_out_hash"][i]),
            int(frames[f"{tag}_tie_mask"][i]))


def _assert_golden(oracle, frames, tag, seed, pal, out, what=""):
    size, pal_hash, out_hash, _ = _golden(frames, tag, seed)
    assert pal.size == size and oracle.hash_words(pal) == pal_hash, (what, tag, seed, "palette")
    assert oracle.hash_words(out) == out_hash, (what, tag, seed, "output")


# ---- 1. frame pipeline: flagged frames among clean ones --------------------------------------------------------------
def _c4_sequence():
    # flagged and clean alternate, so with any lane count a flagged and a clean frame follow each other on some lane
    seq = []
    for f, c in zip(T.C4_FLAGGED, T.C4_CLEAN):
        seq += [("c4", f), ("c4", c)]
    return seq


def _bench_sequence():
    return [("bench", T.BENCH_FLAGGED[0]), ("bench", T.BENCH_CLEAN), ("bench", T.BENCH_FLAGGED[1]), ("bench", T.BENCH_FLAGGED[2])]


def _run_pipeline(dq, pkg, oracle, frames, images, seq, k, lanes, split_ctas, device_frames):
    import torch
    pipe = pkg.FramePipeline(dq.lib, 0, 0 if device_frames else max(images[s].size for s in seq), depth=lanes, split_ctas=split_ctas)
    try:
        assert dq.lib.dq_pipeline_lanes(pipe.handle) == lanes
        cts = [np.zeros(k, np.uint32) for _ in seq]
        nks = [C.c_uint32(k) for _ in seq]
        if device_frames:
            d_in = [torch.from_numpy(images[s].view(np.int32).copy()).cuda() for s in seq]
            d_out = [torch.zeros(images[s].size, dtype=torch.int32, device="cuda") for s in seq]
            torch.cuda.synchronize()
            for i, s in enumerate(seq):
                pipe.submit_device(d_in[i].data_ptr(), d_out[i].data_ptr(), images[s].size, cts[i], nks[i], 0)
            pipe.flush()
            outs = [d.cpu().numpy().view(np.uint32) for d in d_out]
        else:
            ins = [torch.from_numpy(images[s].view(np.int32).copy()).pin_memory() for s in seq]
            outs_t = [torch.zeros(images[s].size, dtype=torch.int32).pin_memory() for s in seq]
            for i in range(len(seq)):
                pipe.submit(ins[i].numpy().view(np.uint32), outs_t[i].numpy().view(np.uint32), k, cts[i], nks[i], 0)
            pipe.flush()
            outs = [o.numpy().view(np.uint32) for o in outs_t]
        what = (lanes, split_ctas, "submit_device" if device_frames else "submit")
        for i, (tag, seed) in enumerate(seq):
            _assert_golden(oracle, frames, tag, seed, cts[i][:nks[i].value], outs[i], what)
        flagged = int(dq.lib.dq_pipeline_flagged_frames(pipe.handle))
        resolved = int(dq.lib.dq_pipeline_resolved_frames(pipe.handle))
        reruns = int(dq.lib.dq_pipeline_rerun_frames(pipe.handle))
        with_mask = sum(1 for tag, seed in seq if _golden(frames, tag, seed)[3] != 0)
        assert with_mask <= flagged <= len(seq), (what, flagged, with_mask)
        # every flagged golden frame is settled by the resolver / a forced cut (as on the default context,
        # test_gpu_frames.py), never by the ordered re-run: these frames have far fewer colours than the re-run's limit, so
        # a re-run would hide a resolver that was skipped or gave up
        assert reruns == 0 and resolved >= with_mask, (what, flagged, resolved, reruns)
        return flagged
    finally:
        pipe.close()


ENV_MODES = {"default": {}, "resolve_large": {"DIVQUANT_B200_RESOLVE": "2"}}


@pytest.mark.parametrize("mode", list(ENV_MODES))
def test_pipeline_flagged_c4_frames(dq, pkg, oracle, frames, images, monkeypatch, mode):
    """Lanes poll quantize_step one phase at a time (resolver and re-split of one lane run while others start frames);
    split kernels run on a share of the SMs.  RESOLVE=2: every flagged rounding goes through the resolver's large form.
    Environment variables are read when the pipeline and its contexts are created."""
    for name, value in ENV_MODES[mode].items():
        monkeypatch.setenv(name, value)
    seq = _c4_sequence()
    counts = {}
    for lanes, split_ctas in ((1, 0), (4, 0), (12, 0), (3, 9)):
        for device_frames in (False, True):
            counts[(lanes, split_ctas, device_frames)] = _run_pipeline(dq, pkg, oracle, frames, images, seq, 64, lanes, split_ctas,
                                                                       device_frames)
    # the audit is a deterministic function of the input (exact integer sums): the same frames are flagged whatever the
    # lane count, SM partition or way of submitting
    assert len(set(counts.values())) == 1, counts


@pytest.mark.parametrize("mode", list(ENV_MODES))
def test_pipeline_flagged_bench_frames(dq, pkg, oracle, frames, images, monkeypatch, mode):
    for name, value in ENV_MODES[mode].items():
        monkeypatch.setenv(name, value)
    seq = _bench_sequence()
    counts = {lanes: _run_pipeline(dq, pkg, oracle, frames, images, seq, 256, lanes, 0, True) for lanes in (1, 12)}
    assert len(set(counts.values())) == 1, counts


# ---- 3. explicit contexts and the SM partition ----------------------------------------------------------------------
@pytest.mark.parametrize("split_ctas", [1, 2, 7, 37, 0])
def test_explicit_context_split_ctas(dq, oracle, frames, images, split_ctas):
    """The resolver names nodes by their ranges of positions, so the partition must not depend on the CTA count."""
    import torch
    lib = dq.lib
    ctx = lib.dq_context_create(0)
    try:
        lib.dq_context_set_split_ctas(ctx, split_ctas)
        for tag, seed in (("c4", 12410), ("c4", 12832), ("c4", 13124), ("bench", 12359)):
            k = 64 if tag == "c4" else 256
            px = images[(tag, seed)]
            d_in = torch.from_numpy(px.view(np.int32).copy()).cuda()
            d_out = torch.empty_like(d_in)
            ct = np.zeros(k, np.uint32)
            nk = C.c_uint32(k)
            torch.cuda.synchronize()
            lib.dq_quant_recurse_device(ctx, px.size, d_in.data_ptr(), d_out.data_ptr(), C.byref(nk), ct.ctypes.data_as(C.POINTER(C.c_uint32)), 0)
            st = dq.last_stats(ctx)
            _assert_golden(oracle, frames, tag, seed, ct[:nk.value], d_out.cpu().numpy().view(np.uint32), split_ctas)
            assert st["tie_flags"] and st["ordered_rerun"] == 0, (split_ctas, seed, st)
            assert st["tie_resolved"] > 0 or st["cut_overrides"] >= 1, (split_ctas, seed, st)
            if seed == T.C4_FORCED:
                assert st["cut_overrides"] >= 1, (split_ctas, seed, st)
    finally:
        lib.dq_context_destroy(ctx)


# ---- 4. quant_varpart_fast with num_bits < 8 / dec_factor > 1 through the resolver ------------------------------------
def _varpart_check(st, entry, what):
    seed, bits, dec, k, int_wrong, forced = entry
    # the device audits a superset of the model's comparisons, and the model flags every input of the table
    assert st["tie_flags"] != 0, (what, st)
    # ... and leaves nothing for the ordered re-run (test_tie_inputs.py: left == 0), so the resolver (with the shift of
    # num_bits and the decimated first-seen sampling) must settle it; the inputs are far below the re-run's limit of
    # colours, so a re-run would hide a resolver that was skipped or gave up
    assert st["ordered_rerun"] == 0 and (st["tie_resolved"] > 0 or st["cut_overrides"] >= 1), (what, st)
    if forced:
        assert st["cut_overrides"] >= 1, (what, st)


def test_varpart_parameters_host_one_row(dq, oracle):
    for entry in T.VARPART_1D:
        seed, bits, dec, k = entry[:4]
        px = oracle.generate(1, 1920, 1080, seed)
        with muted():
            ref, ref_empty = oracle.quant_varpart_fast(px, k, bits, dec)
            pal, empty = dq.quant_varpart_fast(px, k, bits, dec)
        st = dq.last_stats()
        what = ("1d", seed, bits, dec, k)
        assert np.array_equal(pal, ref) and empty == ref_empty, (what, st)
        _varpart_check(st, entry, what)


def test_varpart_parameters_device_2d(dq, oracle):
    import torch
    lib = dq.lib
    ctx = lib.dq_context_create(0)
    try:
        for entry in T.VARPART_2D:
            seed, bits, dec, k = entry[:4]
            px = oracle.generate(1, 1920, 1080, seed)
            with muted():
                ref, ref_empty = oracle.quant_varpart_fast(px, k, bits, dec, rows=1080, cols=1920)
            d_in = torch.from_numpy(px.view(np.int32).copy()).cuda()
            ct = np.zeros(k, np.uint32)
            nk = C.c_uint32(k)
            torch.cuda.synchronize()
            with muted((2,)):
                lib.dq_quant_varpart_device(ctx, px.size, d_in.data_ptr(), 1080, 1920, C.byref(nk), ct.ctypes.data_as(C.POINTER(C.c_uint32)),
                                            bits, dec, 10, 0)
            st = dq.last_stats(ctx)
            what = ("2d", seed, bits, dec, k)
            assert np.array_equal(ct[:nk.value], ref) and k - nk.value == ref_empty, (what, st)
            _varpart_check(st, entry, what)
    finally:
        lib.dq_context_destroy(ctx)


# ---- 5. row sharding on one rank ------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag,seed", [("c4", 12410), ("c4", 12832), ("bench", 12359)])
def test_row_shards_one_rank_flagged(dq, pkg, oracle, frames, images, tag, seed):
    """dq_rows resolves flagged frames like the single-GPU call (merged first-seen indexes, resolver, forced cuts)."""
    import torch
    lib = dq.lib
    k = 64 if tag == "c4" else 256
    px = images[(tag, seed)]
    ctx = lib.dq_context_create(0)
    rows = pkg.RowShards(lib, ctx, None)
    try:
        shard = torch.from_numpy(px.view(np.int32).copy()).cuda()
        out, pal = rows.quant_recurse(shard, px.size, k)
        st = dq.last_stats(ctx)
        _assert_golden(oracle, frames, tag, seed, pal, out.cpu().numpy().view(np.uint32), "dq_rows")
        assert st["tie_flags"] and st["ordered_rerun"] == 0 and (st["tie_resolved"] > 0 or st["cut_overrides"] >= 1), st
        if seed == T.C4_FORCED:
            assert st["cut_overrides"] >= 1, st
    finally:
        rows.close()
        lib.dq_context_destroy(ctx)


# ---- 6. row sharding on 2+ GPUs -------------------------------------------------------------------------------------
def test_row_shards_all_gpus_flagged_frame(built):
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs 2+ GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={min(n, 8)}", "--master-addr",
           "127.0.0.1", "--master-port", str(29300 + os.getpid() % 300), os.path.join(ROOT, "tools", "rows_check.py"),
           "1920", "1080", "64", "1", "12410"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "bit-exact vs single GPU" in res.stdout and "reference fingerprint ok" in res.stdout, res.stdout[-2000:]
