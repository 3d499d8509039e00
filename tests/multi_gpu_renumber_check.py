"""Run under torchrun on >= 2 GPUs: an agent-sharded LargeCrowd with a visible robot, stepped, re-numbered (renumber(): the same
permutation on every rank, the tiles dealt to the ranks when the crowd is a whole number of them) and stepped again with both checks,
must equal one GPU stepping the same crowd, re-numbered the same way, BIT FOR BIT -- over the peer-store exchange on whole tiles
(64 x 64 humans) and over NCCL on a ragged crowd (72 x 72), in fp64 and fp32.  Prints 'MULTI_GPU_RENUMBER_CHECK OK'."""
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

DT, MODEL, ACTION, ROBOT_SAFETY = 0.0125, "hsfm_farina", np.array([0.9, 0.35]), 0.05


def crowd(n_side, dtype, **kw):
    sc = scenarios.jittered_grid_crowd(n_side, pitch=1.0, jitter=0.3, seed=n_side)  # row order: re-numbering changes it
    S, G = sc["states"][0], sc["goals"][0]
    S[:, 5:7] = np.random.RandomState(n_side).uniform(-0.6, 0.6, (S.shape[0], 2))
    robot = np.zeros(13)
    robot[0:2], robot[8], robot[9], robot[12], robot[10:12] = S[:, 0:2].mean(0) + [0.5, 0.5], 0.3, 80.0, 1.0, S[:, 0:2].mean(0) + [4.5, 0.5]
    if dtype == torch.float32:
        S, G, robot = (a.astype(np.float32).astype(np.float64) for a in (S, G, robot))
    return S, G, LargeCrowd(MODEL, S, G, dtype=dtype, robot=robot, robot_safety=ROBOT_SAFETY, consider_robot=True, **kw)


for dtype in (torch.float64, torch.float32):
    for n_side, exchange in ((64, "p2p"), (72, "nccl")):
        S, G, sharded = crowd(n_side, dtype, rank=rank, world=world, exchange=exchange)
        assert sharded.exchange == exchange, (sharded.exchange, getattr(sharded, "_p2p_error", None))
        sharded.step(DT, n_substeps=10, action=ACTION)
        pos = sharded.view[sharded.cur][0:2].double().cpu().numpy().T
        perm = sharded.renumber()
        want = scenarios.spatial_order(pos)
        want = scenarios.deal_tiles(want, world) if len(want) % 128 == 0 else want
        assert np.array_equal(perm, want), f"rank {rank}: permutation ({dtype}, {exchange})"
        sharded.step(DT, n_substeps=10, action=ACTION, pre_checks=True, post_checks=True)
        sharded.check_peers()
        mine = sharded.local_rows(S[perm][sharded.offset:sharded.offset + sharded.n_local])
        mine_flags = (int(sharded.eng.flags[0]), sharded.eng.checks[0].cpu().numpy(), sharded.robot_rows())

        # one GPU: the same 10 sub-steps, the arrays re-numbered by the same permutation, the same 10 sub-steps with the checks
        _, _, single = crowd(n_side, dtype)
        single.step(DT, n_substeps=10, action=ACTION)
        e1 = single.eng
        arrays = [t[..., torch.as_tensor(perm, device=t.device)].clone() for t in (e1.dyn, e1.stat, e1.goals, e1.goal_idx, e1.goal_cnt, single.radius)]
        _, _, ref = crowd(n_side, dtype)
        for t, a in zip((ref.eng.dyn, ref.eng.stat, ref.eng.goals, ref.eng.goal_idx, ref.eng.goal_cnt, ref.radius), arrays):
            t.copy_(a)
        ref.eng.robot.copy_(e1.robot)
        ref.eng.time_now.copy_(e1.time_now)
        ref._publish()
        ref.step(DT, n_substeps=10, action=ACTION, pre_checks=True, post_checks=True)
        want_rows = ref.local_rows(S[perm])[sharded.offset:sharded.offset + sharded.n_local]
        assert np.array_equal(mine, want_rows), f"rank {rank}: sharded re-numbered crowd differs from one GPU ({dtype}, {exchange})"
        assert mine_flags[0] == int(ref.eng.flags[0]) and np.array_equal(mine_flags[1], ref.eng.checks[0].cpu().numpy()), (rank, dtype, exchange)
        assert np.array_equal(mine_flags[2], ref.robot_rows()), (rank, dtype, exchange)
ok = parallel.sum_over_ranks(1.0, "cuda", world)
if rank == 0:
    print(f"MULTI_GPU_RENUMBER_CHECK OK on {int(ok)} ranks")
dist.destroy_process_group()
