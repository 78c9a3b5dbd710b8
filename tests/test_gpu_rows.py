"""GPU test of the pixel-row sharded path (BASELINE.json config 3): histogram per shard, one all-gather of the
(colour, count) lists, merged split replicated on every rank, shard-local remap -- bit-exact against the
single-GPU quant_recurse of the whole image.  Uses as many GPUs as the box has (2+ GPUs go through NCCL)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _run(world, width, height, k):
    script = os.path.join(ROOT, "tools", "rows_check.py")
    if world == 1:
        cmd = [sys.executable, script, str(width), str(height), str(k), "1"]
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
               "127.0.0.1", "--master-port", str(29600 + os.getpid() % 300), script, str(width), str(height), str(k), "1"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "bit-exact vs single GPU" in res.stdout


def test_row_sharded_single_rank(built):
    _run(1, 640, 360, 64)


def test_row_sharded_few_colours_single_rank(built):
    # 320x180 G1 at K=64: the sharded call stays on exact integer sums (it has no ordered path: that needs the whole image
    # in order); rows_check fails if that ever differs from the single-GPU call
    _run(1, 320, 180, 64)


def test_row_sharded_all_gpus(built):
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs 2+ GPUs")
    _run(min(n, 8), 1920, 1080, 256)
