"""Run under torchrun on >= 2 GPUs: an agent-sharded LargeCrowd whose partial sums have slots for only a few units on every rank
(unit_capacity, the finish kernel evaluating the rest) must equal the single-GPU crowd at the default scratch size BIT FOR BIT, over
the peer-store exchange and over NCCL.  Prints 'MULTI_GPU_UNITS_CHECK OK'."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from social_navigation_pyenvs_b200 import scenarios, parallel  # noqa: E402
from social_navigation_pyenvs_b200.large import LargeCrowd  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))

sc = scenarios.jittered_grid_crowd(64, pitch=1.0, jitter=0.3, seed=4)
S0, G0 = sc["states"][0], sc["goals"][0]
S0[:, 5:7] = np.random.RandomState(2).uniform(-0.6, 0.6, (S0.shape[0], 2))
perm = scenarios.spatial_order(S0[:, 0:2])
S, G = np.ascontiguousarray(S0[perm]), np.ascontiguousarray(G0[perm])
for dtype in (torch.float64, torch.float32):
    for exchange in ("p2p", "nccl"):
        sharded = LargeCrowd("hsfm_farina", S, G, dtype=dtype, rank=rank, world=world, exchange=exchange, unit_capacity=3)
        assert sharded.n_local % 128 == 0 and sharded.offset % 128 == 0
        for k in (3, 2):
            sharded.scratch.fill_(0xFF)
            sharded.step(0.0125, n_substeps=k)
            st = sharded.unit_stats()
            assert st["fallback_units"] >= st["max_listed"] - 3 > 0, (rank, st)
        sharded.check_peers()
        mine = sharded.local_rows(S[sharded.offset:sharded.offset + sharded.n_local])
        single = LargeCrowd("hsfm_farina", S, G, dtype=dtype, rank=0, world=1)
        single.step(0.0125, n_substeps=5)
        ref = single.local_rows(S)[sharded.offset:sharded.offset + sharded.n_local]
        assert np.array_equal(mine, ref), f"rank {rank}: sharded crowd with 3 slots differs from the single GPU ({dtype}, {exchange})"
ok = parallel.sum_over_ranks(1.0, "cuda", world)
if rank == 0:
    print(f"MULTI_GPU_UNITS_CHECK OK on {int(ok)} ranks")
dist.destroy_process_group()
