"""Multi-GPU parity of the large crowd's robot (-m gpu, skipped with fewer than two GPUs): tests/multi_gpu_robot_check.py under
torchrun -- the agent-sharded crowd with a visible moving robot and both checks must equal one GPU bit for bit, with the p2p and the
NCCL exchange, and every rank must report the same flags."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs of one node")
@pytest.mark.parametrize("ranks", [2, 8])
def test_sharded_robot_crowd_equals_single_gpu_bit_for_bit(ranks):
    if torch.cuda.device_count() < ranks:
        pytest.skip(f"{ranks} GPUs needed")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={ranks}", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(HERE, "multi_gpu_robot_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and f"MULTI_GPU_ROBOT_CHECK OK on {ranks} ranks" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
