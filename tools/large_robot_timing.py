"""What the robot costs in the large crowd: on the 65536-human hsfm_farina crowd (256 x 256 jittered grid, pitch 2 m, patch order,
as bench.py's 65536_hsfm_single_crowd), in fp64 and fp32, CUDA-event times of

  * a 20-sub-step LargeCrowd.step without a robot;
  * the same step with a visible holonomic robot and both checks (pre_checks, post_checks);
  * the checks alone (a step of 0 sub-steps with both checks);
  * one 360-ray scan (LargeCrowd.scan, 10 m).

Prints one JSON line with the GPU's name and power limit, read in the same run.

    python tools/large_robot_timing.py [--reps 20] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from social_navigation_pyenvs_b200 import scenarios  # noqa: E402
from social_navigation_pyenvs_b200.large import LargeCrowd  # noqa: E402

DT = 0.0125


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + ["?"])[:2] if q.returncode == 0 else (torch.cuda.get_device_name(), "not read")
    return name, power


def time_ms(fn, reps, warmup):
    """Median over `reps` of the CUDA-event time of one call of fn, after `warmup` calls."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return float(np.median(out)), float(np.min(out)), float(np.max(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    sc = scenarios.jittered_grid_crowd(256, pitch=2.0, jitter=0.5, seed=0)
    perm = scenarios.spatial_order(sc["states"][0, :, 0:2])
    S, G = np.ascontiguousarray(sc["states"][0][perm]), np.ascontiguousarray(sc["goals"][0][perm])
    robot = np.zeros(13)
    robot[8], robot[9], robot[12] = 0.3, 80.0, 1.0  # at the origin: between the four humans of the centre
    robot[10:12] = [200.0, 0.0]
    action = np.array([1.0, 0.0])
    name, power = gpu_info()
    result = {"tool": "large_robot_timing", "gpu": name, "power_limit": power, "humans": int(S.shape[0]), "model": "hsfm_farina",
              "order": "patch", "sub_steps_per_step": 20, "scan_rays": 360, "unit": "ms per call (CUDA events; median, min, max)", "reps": args.reps}
    for dtype, tag in ((torch.float64, "f64"), (torch.float32, "f32")):
        bare = LargeCrowd("hsfm_farina", S, G, dtype=dtype)
        withr = LargeCrowd("hsfm_farina", S, G, dtype=dtype, robot=robot, robot_safety=0.0, consider_robot=True)
        result[tag] = {
            "step20_no_robot": time_ms(lambda: bare.step(DT, 20), args.reps, args.warmup),
            "step20_robot_checks": time_ms(lambda: withr.step(DT, 20, action=action, pre_checks=True, post_checks=True), args.reps, args.warmup),
            "checks_only": time_ms(lambda: withr.step(DT, 0, action=action, pre_checks=True, post_checks=True), args.reps, args.warmup),
            "scan_360": time_ms(lambda: withr.scan(2 * np.pi, 360, 10.0), args.reps, args.warmup),
        }
        del bare, withr
        torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
