"""Dev tool: what ONE rank of an 8-way agent-sharded 65536 crowd executes per sub-step, on one GPU (the rest of the crowd frozen).
Run under ncu for the per-kernel durations:  ncu --metrics gpu__time_duration.sum --csv ... python tools/diag_large_shard.py 8 3"""
import sys, os
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from social_navigation_pyenvs_b200 import scenarios
from social_navigation_pyenvs_b200.large import LargeCrowd

ways, rank = int(sys.argv[1]), int(sys.argv[2])
sc = scenarios.jittered_grid_crowd(256, pitch=2.0, jitter=0.5, seed=0)
perm = scenarios.spatial_order(sc["states"][0, :, 0:2])
if os.environ.get("SNP_LARGE_DEAL", "1") == "1":  # the bench's load balancing: 128-human tiles dealt round-robin to the ranks
    perm = scenarios.deal_tiles(perm, ways)
S, G = np.ascontiguousarray(sc["states"][0, perm]), np.ascontiguousarray(sc["goals"][0, perm])
n = S.shape[0] // ways
crowd = LargeCrowd("hsfm_farina", S, G, dtype=torch.float64, shard=(rank * n, n))
# a slice recomputes the tile boxes of the view it reads every sub-step (in a real sharded run the other ranks' producers write the
# boxes of their tiles; here the rest of the crowd is frozen and nobody would): one launch more than a rank of a sharded run
for _ in range(2):
    crowd.step(0.0125, 1)
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(10):
    crowd.step(0.0125, 1)
b.record(); torch.cuda.synchronize()
print(f"{ways}-way shard, rank {rank}: {a.elapsed_time(b) / 10:.4f} ms per sub-step ({crowd.exchange})")
