"""What the policies' lookahead costs beyond one CTA per env: snp_lookahead (TiledCrowdEngine.lookahead_from on the constant-velocity
propagation of the crowd, 81 actions, 13 values per row) for E x N = 64 x 1024, 16 x 4096 and 1 x 65 536 in fp64 and fp32 -- all of
them run the human-split kernel except 64 x 1024 fp32, which one CTA per env still holds -- and 64 x 600 in fp64 with the whole-env
kernel (the default there) against the forced split: the numbers for where the selection between the two should sit.

Each shape: the CUDA-event time of one snp_lookahead call (median, min, max of --reps after --warmup) and of a plain fill_ of the same
rotated buffer in the same run, and bytes written (rotated + rewards) / time for both.  Every output exceeds the 126 MB of L2.
Prints one JSON line with the GPU's name and power limit, read in the same run.

    python tools/large_lookahead_timing.py [--reps 20] [--warmup 3]
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
from social_navigation_pyenvs_b200 import TiledCrowdEngine, scenarios  # noqa: E402

DT = 0.25
MODEL = "hsfm_farina"
SHAPES = ((64, 1024), (16, 4096), (1, 65536))


def actions():
    speeds = [(np.exp((i + 1) / 5) - 1) / (np.e - 1) for i in range(5)]
    rot = np.linspace(0, 2 * np.pi, 16, endpoint=False)
    return np.array([[0.0, 0.0]] + [[s * np.cos(r), s * np.sin(r)] for r in rot for s in speeds])


def envs(E, N):
    side = int(np.ceil(np.sqrt(N)))
    S, G = [], []
    for e in range(E):
        sc = scenarios.jittered_grid_crowd(side, pitch=1.0, jitter=0.3, seed=e)
        S.append(sc["states"][0][:N]); G.append(sc["goals"][0][:N])
    robots = np.zeros((E, 13))
    robots[:, 0] = 0.5
    robots[:, 8], robots[:, 9], robots[:, 12] = 0.3, 80.0, 1.0
    robots[:, 10:12] = [200.0, 0.0]
    return np.stack(S), np.stack(G), robots


def measure(eng, nxt, reps, warmup, split=False):
    rot, rew = eng.lookahead_from(nxt, DT, yaw_from_next=True, split_humans=split)
    nbytes = rot.numel() * rot.element_size() + rew.numel() * rew.element_size()
    look = time_ms(lambda: eng.lookahead_from(nxt, DT, yaw_from_next=True, split_humans=split), reps, warmup)
    fill = time_ms(lambda: rot.fill_(0.0), reps, warmup)
    gbs = lambda ms: nbytes / (ms * 1e-3) / 1e9
    return {"bytes": nbytes, "lookahead_ms": look, "fill_ms": fill, "lookahead_GBps": gbs(look[0]), "fill_GBps": gbs(fill[0]),
            "lookahead_over_fill": fill[0] / look[0]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the timing needs a GPU"
    name, power = gpu_info()
    result = {"tool": "large_lookahead_timing", "gpu": name, "power_limit": power, "model": MODEL, "actions": 81, "values_per_row": 13,
              "unit": "ms per call (CUDA events; median, min, max); GB/s = bytes written / median", "reps": args.reps,
              "fill": "torch fill_ of the rotated buffer, same run", "sms": torch.cuda.get_device_properties(0).multi_processor_count}
    cases = [(E, N, dtype, False) for E, N in SHAPES for dtype in (torch.float64, torch.float32)]
    cases += [(64, 600, torch.float64, False), (64, 600, torch.float64, True)]
    for E, N, dtype, split in cases:
        key = f"{E}x{N}_{'f64' if dtype == torch.float64 else 'f32'}" + ("_forced_split" if split else "")
        S, G, robots = envs(E, N)
        eng = TiledCrowdEngine.from_reference_arrays(MODEL, S, G, robot=robots, dtype=dtype)
        eng.set_action_space(actions())
        nxt = eng.constant_velocity_next(DT)
        out = measure(eng, nxt, args.reps, args.warmup, split)
        result[key] = out
        print(json.dumps({key: out}), file=sys.stderr, flush=True)
        del eng, nxt
        torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
