"""Re-numbering an agent-sharded crowd (-m gpu, skipped with fewer than two GPUs): tests/multi_gpu_renumber_check.py under torchrun --
renumber() and further steps on 2 and 8 ranks equal one GPU stepping the crowd re-numbered the same way, bit for bit, over the
peer-store exchange on whole tiles and over NCCL on a ragged crowd."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs of one node")
@pytest.mark.parametrize("ranks", [2, 8])
def test_sharded_renumber_equals_single_gpu_bit_for_bit(ranks):
    if torch.cuda.device_count() < ranks:
        pytest.skip(f"{ranks} GPUs needed")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={ranks}", "--master-addr", "127.0.0.1",
           "--master-port", "29537", os.path.join(HERE, "multi_gpu_renumber_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and f"MULTI_GPU_RENUMBER_CHECK OK on {ranks} ranks" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
