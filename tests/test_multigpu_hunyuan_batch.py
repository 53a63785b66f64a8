"""Ulysses on real GPUs at batch 2 with per-sample text lengths: N-GPU result == 1-GPU result, bit for bit (needs >= 2
B200s; skipped otherwise)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("world", [2, 4])
def test_hunyuan_batch2_sequence_parallel_equals_single_gpu(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(29700 + world),
           os.path.join(ROOT, "tests", "mgpu_hunyuan_batch.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, VB_ULYSSES="nccl"))
    print(res.stdout[-3000:])
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "MISMATCH" not in res.stdout and "bit-identical" in res.stdout
