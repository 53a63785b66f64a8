"""Ulysses on real GPUs: N-GPU result == 1-GPU result (needs >= 2 B200s; skipped otherwise)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("mode", ["peer", "peer-split", "nccl", "nccl-contiguous"])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_sequence_parallel_equals_single_gpu(world, mode):
    """mode "peer": exchange fused into the kernels over NVLink peer memory; "nccl": all-to-all collectives;
    "peer-split": query-half units even at 2 ranks; "-contiguous": the reference's contiguous head chunks instead of the
    cost-balanced placement."""
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    exchange = mode.split("-")[0]
    port = 29600 + world + (10 if exchange == "nccl" else 0) + (20 if mode.endswith("-contiguous") else 0) \
        + (40 if mode == "peer-split" else 0)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "mgpu_check.py"), mode]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, VB_ULYSSES=exchange))
    print(res.stdout[-3000:])
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "MISMATCH" not in res.stdout
    if exchange == "peer":
        assert "peer-memory exchange unavailable" not in res.stdout
