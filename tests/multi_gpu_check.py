"""Run under torchrun on >= 2 GPUs: agent-sharded LargeCrowd must equal the single-GPU result BIT FOR BIT (each agent's
j-ascending pair loop is identical, only the owner of the row changes), and env-sharded engines must equal the slices of one
big engine.  Prints 'MULTI_GPU_CHECK OK'."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from social_navigation_pyenvs_b200 import CrowdEngine, scenarios, parallel  # noqa: E402
from social_navigation_pyenvs_b200.large import LargeCrowd  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
sc_env = scenarios.circular_crossing(64, 7, seed0=300)  # before CUDA init (forks workers only for >= 256 envs)
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))

# ---- one crowd sharded by agent ----
sc = scenarios.jittered_grid_crowd(32, pitch=1.0, jitter=0.3, seed=1)
S, G = sc["states"][0], sc["goals"][0]
rng = np.random.RandomState(0)
S[:, 5:7] = rng.uniform(-0.5, 0.5, (S.shape[0], 2))
# exchange "p2p" = the whole sub-step loop in one C call (snp_large_run_p2p: producer stores entries + tile boxes into every rank's
# next view, device-side barrier kernel); "nccl" = one call per sub-step, then an all-gather.  The single-GPU crowd is run both
# through the fused call and, with "nccl" forced, one call per sub-step.
for dtype, exchange in ((torch.float64, "nccl"), (torch.float32, "nccl"), (torch.float64, "p2p"), (torch.float32, "p2p")):
    sharded = LargeCrowd("hsfm_new_guo", S, G, dtype=dtype, rank=rank, world=world, exchange=exchange)
    assert sharded.exchange == exchange
    sharded.step(0.0125, n_substeps=3)
    sharded.step(0.0125, n_substeps=2)   # a second call continues from the other view buffer with a later barrier epoch
    sharded.check_peers()
    mine = sharded.local_rows(S[sharded.offset:sharded.offset + sharded.n_local])
    for single_exchange in ("fused", "nccl"):
        single = LargeCrowd("hsfm_new_guo", S, G, dtype=dtype, rank=0, world=1, exchange={"fused": "auto", "nccl": "nccl"}[single_exchange])
        assert single.exchange == single_exchange
        single.step(0.0125, n_substeps=5)
        ref = single.local_rows(S)[sharded.offset:sharded.offset + sharded.n_local]
        assert np.array_equal(mine, ref), f"rank {rank}: sharded crowd differs from single-GPU crowd ({dtype}, {exchange}, single {single_exchange})"


# ---- a ragged crowd sharded by agent: 5184 humans, 2592 per rank on 2 ranks and 648 on 8 -- not whole tiles, so the ranks exchange
# over NCCL, and rank 0's slice starts on a tile and ends inside one that also holds rank 1's humans.  Scratch and tile boxes are
# poisoned before every call, so a partial sum the sub-step did not write shows up as NaN. ----
def poisoned_step(crowd, k):
    crowd.scratch.fill_(0xFF)
    for v in crowd._vbuf:
        boxes = v[5 * crowd.n_total:].view(crowd._n_tiles, 5)
        boxes[:, :4] = 1e30
        boxes[:, 4] = 0.0
    crowd.step(0.0125, n_substeps=k)


sc = scenarios.jittered_grid_crowd(72, pitch=1.0, jitter=0.3, seed=3)
S0, G0 = sc["states"][0], sc["goals"][0]
S0[:, 5:7] = np.random.RandomState(1).uniform(-0.6, 0.6, (S0.shape[0], 2))
for order in ("row", "patch"):
    perm = scenarios.spatial_order(S0[:, 0:2]) if order == "patch" else np.arange(S0.shape[0])
    S, G = np.ascontiguousarray(S0[perm]), np.ascontiguousarray(G0[perm])
    for dtype in (torch.float64, torch.float32):
        sharded = LargeCrowd("hsfm_farina", S, G, dtype=dtype, rank=rank, world=world)
        assert sharded.exchange == "nccl" and sharded.n_local % 128 != 0
        poisoned_step(sharded, 3)
        poisoned_step(sharded, 2)
        mine = sharded.local_rows(S[sharded.offset:sharded.offset + sharded.n_local])
        single = LargeCrowd("hsfm_farina", S, G, dtype=dtype, rank=0, world=1)
        poisoned_step(single, 5)
        ref = single.local_rows(S)[sharded.offset:sharded.offset + sharded.n_local]
        assert np.array_equal(mine, ref), f"rank {rank}: ragged sharded crowd differs from single-GPU crowd ({dtype}, {order} order)"

# ---- independent envs sharded by env: no collective on the data path ----
states = np.concatenate([sc_env["states"], sc_env["robot"][:, None]], 1)
sl = parallel.env_shard(64, rank, world)
part = CrowdEngine.from_reference_arrays("hsfm_farina", states[sl], sc_env["goals"][sl], consider_robot=True)
part.step(np.tile([0.0, 1.0], (sl.stop - sl.start, 1)), n_substeps=20)
full = CrowdEngine.from_reference_arrays("hsfm_farina", states, sc_env["goals"], consider_robot=True)
full.step(np.tile([0.0, 1.0], (64, 1)), n_substeps=20)
assert np.array_equal(part.rows(states[sl]), full.rows(states)[sl]), f"rank {rank}: env shard differs"
assert np.array_equal(part.flags.cpu().numpy(), full.flags.cpu().numpy()[sl])
ok = parallel.sum_over_ranks(1.0, "cuda", world)
if rank == 0:
    print(f"MULTI_GPU_CHECK OK on {int(ok)} ranks")
dist.destroy_process_group()
