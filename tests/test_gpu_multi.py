"""Multi-GPU parity (-m gpu, skipped with fewer than two GPUs): tests/multi_gpu_check.py under torchrun -- the agent-sharded
LargeCrowd (fused peer-store exchange, NCCL all-gather) must equal the single-GPU crowd -- stepped in one call or one call per sub-step
with the all-gather -- BIT FOR BIT, and env-sharded engines the slices of one big engine.  A ragged crowd (72 x 72 = 5184 humans,
row and patch order, fp64 and fp32) splits into slices that are not whole 128-human tiles, so its ranks exchange over NCCL and
rank 0's slice ends inside a tile shared with rank 1; its scratch is poisoned before every call."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs of one node")
@pytest.mark.parametrize("ranks", [2, 8])
def test_sharded_results_equal_single_gpu_bit_for_bit(ranks):
    if torch.cuda.device_count() < ranks:
        pytest.skip(f"{ranks} GPUs needed")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={ranks}", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(HERE, "multi_gpu_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and f"MULTI_GPU_CHECK OK on {ranks} ranks" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
