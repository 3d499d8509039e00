"""How much a long run of the large crowd slows down as its humans mix, and what re-numbering it now and then (LargeCrowd.renumber)
wins back.  hsfm_farina, one GPU, the bench's 65,536-human jittered grid (pitch 2 m) numbered patch by patch, in two variants:

  * "mirrored": the bench's goals, every human walking through the crowd's centre to its mirror point (and back);
  * "mixing":   every human walking to the start of a seeded random other human (and back to its own): strong mixing.

For each variant and dtype, two crowds start from the same state with unit_capacity="auto": one is never re-numbered, the other is
re-numbered every --every sub-steps.  Both run --substeps sub-steps in calls of --call, their calls alternated.  Every --every
sub-steps the tool reports, for both: ms per sub-step (CUDA events, mean over the window's calls), the most (agent block, entity
chunk) units in reach one sub-step listed (unit_stats()["max_listed"]) and the capacity "auto" has reached.  Also the time of
one renumber() (host clock around the call, which ends in a device synchronisation; median).

Prints one JSON line per window and a final JSON result with the GPU's name and power limit, read in the same run.

    python tools/large_renumber_timing.py [--substeps 4000] [--call 20] [--every 200] [--dtypes f64,f32] [--out FILE]
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
from large_robot_timing import gpu_info  # noqa: E402
from social_navigation_pyenvs_b200 import scenarios  # noqa: E402
from social_navigation_pyenvs_b200.large import LargeCrowd  # noqa: E402

DT = 0.0125
MODEL = "hsfm_farina"


def crowd_rows(goals):
    sc = scenarios.jittered_grid_crowd(256, pitch=2.0, jitter=0.5, seed=0)
    S, G = sc["states"][0], sc["goals"][0]
    if goals == "mixing":
        other = np.random.RandomState(1).permutation(len(S))
        G[:, 0], G[:, 1] = S[other, 0:2], S[:, 0:2]
        S[:, 10:12] = G[:, 0]
    perm = scenarios.spatial_order(S[:, 0:2])
    return np.ascontiguousarray(S[perm]), np.ascontiguousarray(G[perm])


def call_ms(crowd, k):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    crowd.step(DT, n_substeps=k)
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def run(goals, dtype, args):
    S, G = crowd_rows(goals)
    plain = LargeCrowd(MODEL, S, G, dtype=dtype, unit_capacity="auto")
    renum = LargeCrowd(MODEL, S, G, dtype=dtype, unit_capacity="auto")
    warm = LargeCrowd(MODEL, S, G, dtype=dtype, unit_capacity="auto")  # loads the modules; the two runs start from the same state
    warm.step(DT, n_substeps=args.call)
    warm.renumber()
    del warm
    windows, renumber_ms, done = [], [], 0
    while done < args.substeps:
        t = {"plain": [], "renumbered": []}
        for _ in range(args.every // args.call):
            t["plain"].append(call_ms(plain, args.call) / args.call)
            t["renumbered"].append(call_ms(renum, args.call) / args.call)
        done += args.every
        row = {"goals": goals, "dtype": str(dtype).split(".")[1], "substeps": done}
        for tag, c in (("plain", plain), ("renumbered", renum)):
            st = c.unit_stats()
            row[tag] = {"ms_per_substep": round(float(np.mean(t[tag])), 4), "units_listed": st["max_listed"], "capacity": st["capacity"]}
        print(json.dumps(row), flush=True)
        windows.append(row)
        if done < args.substeps:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            renum.renumber()
            renumber_ms.append((time.perf_counter() - t0) * 1e3)
    return {"windows": windows, "renumber_ms_median": round(float(np.median(renumber_ms)), 3),
            "renumber_ms_first": round(renumber_ms[0], 3), "units_all": (len(S) // 128) ** 2}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--substeps", type=int, default=4000)
    ap.add_argument("--call", type=int, default=20)
    ap.add_argument("--every", type=int, default=200)
    ap.add_argument("--dtypes", default="f64,f32")
    ap.add_argument("--goals", default="mirrored,mixing")
    ap.add_argument("--out", help="also write the result as JSON to this file")
    args = ap.parse_args()
    assert args.every % args.call == 0 and args.substeps % args.every == 0
    assert torch.cuda.is_available(), "large_renumber_timing measures on a GPU"
    name, power = gpu_info()
    result = {"tool": "large_renumber_timing", "gpu": name, "power_limit": power, "model": MODEL, "humans": 65536,
              "substeps": args.substeps, "call": args.call, "every": args.every}
    for goals in args.goals.split(","):
        for tag in args.dtypes.split(","):
            result[f"{goals}_{tag}"] = run(goals, torch.float64 if tag == "f64" else torch.float32, args)
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({k: v for k, v in result.items() if not isinstance(v, dict)} |
                     {k: {"renumber_ms_median": v["renumber_ms_median"], "first": v["windows"][0], "last": v["windows"][-1]}
                      for k, v in result.items() if isinstance(v, dict)}))


if __name__ == "__main__":
    main()
