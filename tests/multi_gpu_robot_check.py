"""Run under torchrun on >= 2 GPUs: the agent-sharded LargeCrowd with a robot (visible, holonomic and unicycle, both checks) must
equal the single-GPU crowd BIT FOR BIT -- the humans, the robot, the clock and the flags / checks, on every rank -- with the p2p
(peer-store) and the NCCL exchange, and with a ragged crowd whose ranks exchange over NCCL.  Prints 'MULTI_GPU_ROBOT_CHECK OK'."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from social_navigation_pyenvs_b200 import scenarios  # noqa: E402
from social_navigation_pyenvs_b200.large import LargeCrowd  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))

ROBOT = np.zeros(13)
ROBOT[0:2], ROBOT[2], ROBOT[8], ROBOT[9], ROBOT[12], ROBOT[10:12] = [0.5, 0.5], 0.3, 0.3, 80.0, 1.0, [6.0, 2.0]
KEYS = ("collision", "dmin", "reaching_goal", "reward", "terminated", "truncated", "info", "actual_collision", "actual_dmin", "actual_goal")


def run(crowd, kinematics, action):
    for _ in range(2):
        crowd.step(0.0125, n_substeps=3, action=action, kinematics=kinematics, pre_checks=True, post_checks=True)
    crowd.check_peers()
    f = crowd.decode_flags()
    return crowd.robot_rows(), float(crowd.eng.time_now[0]), np.array([float(f[k][0]) for k in KEYS])


def compare(S, G, dtype, exchange, label):
    for kinematics, action in (("holonomic", [0.8, 0.3]), ("unicycle", [0.8, 0.05])):
        kw = dict(dtype=dtype, robot=ROBOT, robot_safety=0.05, consider_robot=True)
        sharded = LargeCrowd("hsfm_farina", S, G, rank=rank, world=world, exchange=exchange, **kw)
        assert exchange == "auto" or sharded.exchange == exchange, (sharded.exchange, exchange)
        rb, t, fl = run(sharded, kinematics, action)
        mine = sharded.local_rows(S[sharded.offset:sharded.offset + sharded.n_local])
        single = LargeCrowd("hsfm_farina", S, G, **kw)
        rb1, t1, fl1 = run(single, kinematics, action)
        ref = single.local_rows(S)[sharded.offset:sharded.offset + sharded.n_local]
        what = f"rank {rank}: {label} {dtype} {kinematics}"
        assert np.array_equal(mine, ref), what + ": humans differ from one GPU"
        assert np.array_equal(rb, rb1) and t == t1, what + ": robot / clock differ from one GPU"
        assert np.array_equal(fl, fl1), what + ": flags / checks differ from one GPU"
        every = [None] * world
        dist.all_gather_object(every, fl.tolist())
        assert all(e == every[0] for e in every), what + ": ranks disagree on the flags"


sc = scenarios.jittered_grid_crowd(32, pitch=1.0, jitter=0.3, seed=1)
S, G = sc["states"][0], sc["goals"][0]
S[:, 5:7] = np.random.RandomState(0).uniform(-0.5, 0.5, (S.shape[0], 2))
for dtype in (torch.float64, torch.float32):
    for exchange in ("p2p", "nccl"):
        compare(S, G, dtype, exchange, "1024 humans")

# ragged: 5184 humans, slices that are not whole tiles -> NCCL
sc = scenarios.jittered_grid_crowd(72, pitch=1.0, jitter=0.3, seed=3)
S, G = sc["states"][0], sc["goals"][0]
S[:, 5:7] = np.random.RandomState(1).uniform(-0.6, 0.6, (S.shape[0], 2))
for dtype in (torch.float64, torch.float32):
    compare(S, G, dtype, "auto", "5184 humans")

dist.barrier()
if rank == 0:
    print(f"MULTI_GPU_ROBOT_CHECK OK on {world} ranks")
dist.destroy_process_group()
