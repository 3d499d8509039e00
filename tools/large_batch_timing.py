"""What a batch of large crowds costs: E environments of N humans (hsfm_farina, E seeded jittered grids of pitch 1 m around the
example walls, a visible holonomic robot per env, both checks, 20 sub-steps per call), in fp64 and fp32, CUDA-event times of

  * one TiledCrowdEngine.step (snp_large_batch_step: all E envs in one call);
  * the loop it replaces: E LargeCrowd.step calls, one per env;
  * at N = 512 also CrowdEngine.step (snp_step's block-packed kernel) on the same envs: where the two engines cross over.

E x N = 64 x 1024, 16 x 4096, 4 x 16384 and 64 x 512.  Prints one JSON line with the GPU's name and power limit, read in the same run.

    python tools/large_batch_timing.py [--reps 20] [--warmup 3]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from large_robot_timing import gpu_info, time_ms  # noqa: E402
from social_navigation_pyenvs_b200 import CrowdEngine, TiledCrowdEngine, scenarios  # noqa: E402
from social_navigation_pyenvs_b200.large import LargeCrowd  # noqa: E402

DT = 0.0125
MODEL = "hsfm_farina"
SHAPES = ((64, 1024), (16, 4096), (4, 16384), (64, 512))


def envs(E, N):
    side = int(np.ceil(np.sqrt(N)))
    S, G = [], []
    for e in range(E):
        sc = scenarios.jittered_grid_crowd(side, pitch=1.0, jitter=0.3, seed=e)
        S.append(sc["states"][0][:N]); G.append(sc["goals"][0][:N])
    S, G = np.stack(S), np.stack(G)
    robots = np.zeros((E, 13))
    robots[:, 0] = 0.5
    robots[:, 8], robots[:, 9], robots[:, 12] = 0.3, 80.0, 1.0
    robots[:, 10:12] = [200.0, 0.0]
    return S, G, robots


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    walls = scenarios.pack_walls(scenarios.EXAMPLE_WALLS)
    name, power = gpu_info()
    result = {"tool": "large_batch_timing", "gpu": name, "power_limit": power, "model": MODEL, "walls": "example", "robot": "visible holonomic",
              "checks": "pre + post", "sub_steps_per_call": 20, "unit": "ms per call (CUDA events; median, min, max)", "reps": args.reps}
    for E, N in SHAPES:
        S, G, robots = envs(E, N)
        action = np.tile([1.0, 0.0], (E, 1))
        for dtype, tag in ((torch.float64, "f64"), (torch.float32, "f32")):
            key = f"{E}x{N}_{tag}"
            batch = TiledCrowdEngine.from_reference_arrays(MODEL, S, G, walls=walls, robot=robots, dtype=dtype)
            batch.consider_robot = True
            out = {"batch": time_ms(lambda: batch.step(action, DT, 20, pre_checks=True, post_checks=True), args.reps, args.warmup)}
            del batch
            if N > 512:
                loop = [LargeCrowd(MODEL, S[e], G[e], walls=walls, dtype=dtype, robot=robots[e], consider_robot=True) for e in range(E)]

                def run_loop():
                    for e, one in enumerate(loop):
                        one.step(DT, 20, action=action[e], pre_checks=True, post_checks=True)
                out["loop_of_large_crowds"] = time_ms(run_loop, args.reps, args.warmup)
                out["speedup_over_loop"] = out["loop_of_large_crowds"][0] / out["batch"][0]
                del loop
            else:
                small = CrowdEngine.from_reference_arrays(MODEL, np.concatenate([S, robots[:, None]], 1), G, walls=walls, consider_robot=True, dtype=dtype)
                out["crowd_engine"] = time_ms(lambda: small.step(action, DT, 20, pre_checks=True, post_checks=True), args.reps, args.warmup)
                del small
            result[key] = out
            torch.cuda.empty_cache()
            print(json.dumps({key: out}), file=sys.stderr, flush=True)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
