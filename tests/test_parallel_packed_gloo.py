"""all_gather_columns_packed on CPU with the gloo backend, world_size 2: buffers of three dtypes (the per-agent arrays a re-numbering
of a sharded crowd gathers) travel in one collective and land bit for bit in every rank's columns."""
import os

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from social_navigation_pyenvs_b200 import parallel


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        N = 96
        full = [torch.randn((10, N), generator=torch.Generator().manual_seed(1), dtype=torch.float64),
                torch.randn((4, N), generator=torch.Generator().manual_seed(2)).to(torch.float32),
                torch.randint(-5, 5, (2, N), generator=torch.Generator().manual_seed(3), dtype=torch.int32)]
        full[0][3, 7] = float("nan")
        off, n = parallel.agent_shard(N, rank, world)
        bufs = [torch.full_like(f, -1) for f in full]
        for b, f in zip(bufs, full):
            b[:, off:off + n] = f[:, off:off + n]  # only the own columns are valid
        parallel.all_gather_columns_packed(bufs, off, n, world)
        out[rank] = all(torch.equal(b.view(torch.uint8), f.view(torch.uint8)) for b, f in zip(bufs, full))
    finally:
        dist.destroy_process_group()


def test_packed_gather_of_mixed_dtypes_world_size_2():
    world = 2
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(world, 29737, out), nprocs=world, join=True)
        assert dict(out) == {0: True, 1: True}
