"""Timing of the batched gym beyond 512 humans per env, one GPU, fp64, circle crossing:

  * the on-device reset (snp_reset) at E x N = 64 x 1024 with the warp kernel and with the CTA kernel forced (SNP_RESET_FORCE_CTA),
    and at 16 x 4096 and 4 x 6000 (CTA kernel); circle_radius = N, so the rejection sampler finishes in few attempts;
  * a loop of --steps gym steps (BatchedSocialNavGym.step, hsfm_farina, visible robot) at 64 x 1024, circle_radius 512, with and
    without spatial_order (the patch-by-patch re-numbering after the reset).

Reset: median CUDA-event time of one reset_scenario call over --reps, after a warm-up call.  Gym loop: host clock around the whole
loop, which ends in the device synchronisation of the observation's copy (every step returns its observation to the host), and the
mean ms per step.  Prints one JSON line per measurement and a final JSON result with the GPU's name and power limit, read in the
same run.

    python tools/large_gym_timing.py [--steps 100] [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from large_robot_timing import gpu_info, time_ms  # noqa: E402
from social_navigation_pyenvs_b200 import TiledCrowdEngine  # noqa: E402
from social_navigation_pyenvs_b200.social_nav_gym import BatchedSocialNavGym  # noqa: E402


def reset_ms(E, N, force_cta, reps):
    eng = TiledCrowdEngine("hsfm_farina", E, N, G=2, has_robot=True)
    return time_ms(lambda: eng.reset_scenario("circle_crossing", seed0=2000, circle_radius=float(N), force_cta=force_cta), reps, 1)[0]


def gym_loop_ms(E, N, spatial_order, steps):
    g = BatchedSocialNavGym(E)
    g.configure(dict(human_policy="hsfm_farina", human_num=N, circle_radius=N / 2, robot_visible=True, spatial_order=spatial_order))
    g.reset("train", test_case=0)
    act = np.tile([0.0, 1.0], (E, 1))
    g.step(act)  # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        g.step(act)
    return (time.perf_counter() - t0) * 1e3 / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("large_gym_timing: needs a CUDA device")
    name, power = gpu_info()
    lines = []
    for E, N, kernels in [(64, 1024, ("warp", "cta")), (16, 4096, ("cta",)), (4, 6000, ("cta",))]:
        for k in kernels:
            ms = reset_ms(E, N, k == "cta", args.reps)
            lines.append(dict(what="reset", E=E, N=N, kernel=k, ms=round(ms, 3)))
            print(json.dumps(lines[-1]), flush=True)
    for so in (False, True):
        ms = gym_loop_ms(64, 1024, so, args.steps)
        lines.append(dict(what="gym_step", E=64, N=1024, spatial_order=so, steps=args.steps, ms_per_step=round(ms, 3)))
        print(json.dumps(lines[-1]), flush=True)
    result = dict(gpu=name, power_limit=power, dtype="f64", lines=lines)
    print(json.dumps(result))
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(result) + "\n")


if __name__ == "__main__":
    main()
