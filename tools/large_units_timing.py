"""What the unit-sized scratch of the large crowd (LargeCrowd(unit_capacity=...), SNP_OPT_UNIT_SCRATCH) costs and saves, hsfm_farina,
one GPU, jittered grids of pitch 2 m numbered patch by patch (the bench's crowd at 65,536), CUDA-event times (median of --reps calls of
--substeps sub-steps each, after --warmup calls):

  * 65,536 humans, fp64 and fp32: the default scratch against a capacity of 1.25 x the units listed, the two alternated call by call,
    with the units listed and both scratch sizes;
  * the same crowd at capacity 0: every unit evaluated by the finish kernel (the fallback's cost);
  * 262,144 / 1,048,576 / 1,500,625 / 4,000,000 humans in fp64 with unit_capacity="auto": scratch bytes and ms per sub-step, the
    default scratch's size beside it, and its time where it fits in 60 % of the card.

Prints one JSON line with the GPU's name and power limit, read in the same run.

    python tools/large_units_timing.py [--reps 20] [--warmup 3] [--substeps 10] [--sizes 512,1024,1225,2000] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from large_robot_timing import gpu_info  # noqa: E402
from social_navigation_pyenvs_b200 import _lib as L, scenarios  # noqa: E402
from social_navigation_pyenvs_b200.large import LargeCrowd  # noqa: E402

DT = 0.0125
MODEL = "hsfm_farina"


def crowd_rows(side, seed=0):
    sc = scenarios.jittered_grid_crowd(side, pitch=2.0, jitter=0.5, seed=seed)
    perm = scenarios.spatial_order(sc["states"][0, :, 0:2])
    return np.ascontiguousarray(sc["states"][0][perm]), np.ascontiguousarray(sc["goals"][0][perm])


def one_call_ms(crowd, k):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    crowd.step(DT, n_substeps=k)
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def alternated(crowds, k, reps, warmup):
    """Median ms per sub-step of each crowd, their calls alternated."""
    for _ in range(warmup):
        for c in crowds:
            c.step(DT, n_substeps=k)
    torch.cuda.synchronize()
    times = [[] for _ in crowds]
    for _ in range(reps):
        for t, c in zip(times, crowds):
            t.append(one_call_ms(c, k) / k)
    return [round(float(np.median(t)), 4) for t in times]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--substeps", type=int, default=10)
    ap.add_argument("--sizes", default="512,1024,1225,2000")
    ap.add_argument("--out", help="also write the result as JSON to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "large_units_timing measures on a GPU"
    name, power = gpu_info()
    total = torch.cuda.get_device_properties(0).total_memory
    lib = L.lib()
    result = {"tool": "large_units_timing", "gpu": name, "power_limit": power, "model": MODEL, "crowd": "jittered grid, pitch 2 m, patch order",
              "unit": "ms per sub-step (CUDA events, median)", "reps": args.reps, "substeps_per_call": args.substeps}
    S, G = crowd_rows(256)
    n = S.shape[0]
    for dtype, tag in ((torch.float64, "f64"), (torch.float32, "f32")):
        dt = L.SNP_F64 if tag == "f64" else L.SNP_F32
        default = LargeCrowd(MODEL, S, G, dtype=dtype)
        probe = LargeCrowd(MODEL, S, G, dtype=dtype, unit_capacity=(n // 128) ** 2)  # a slot for every unit: what a step lists
        probe.step(DT, n_substeps=args.substeps)
        listed = probe.unit_stats()["max_listed"]
        del probe
        cap = -(-5 * listed // 4)
        sized = LargeCrowd(MODEL, S, G, dtype=dtype, unit_capacity=cap)
        none = LargeCrowd(MODEL, S, G, dtype=dtype, unit_capacity=0)
        ms_default, ms_sized = alternated([default, sized], args.substeps, args.reps, args.warmup)
        (ms_none,) = alternated([none], args.substeps, max(5, args.reps // 4), 1)
        assert sized.unit_stats()["fallback_units"] == 0
        result[f"65536_{tag}"] = {"units_listed": listed, "units_all": (n // 128) ** 2, "capacity": cap,
                                  "scratch_bytes_default": int(lib.snp_large_scratch_bytes(n, n, dt)), "scratch_bytes_capacity": sized.scratch.numel(),
                                  "ms_default": ms_default, "ms_capacity": ms_sized,
                                  "ms_capacity_0": ms_none, "fallback_units_per_call_at_0": none.unit_stats()["fallback_units"]}
        print(json.dumps({f"65536_{tag}": result[f"65536_{tag}"]}), flush=True)
        del default, sized, none
        torch.cuda.empty_cache()
    for side in (int(s) for s in args.sizes.split(",")):
        S, G = crowd_rows(side)
        n = S.shape[0]
        if side == 2000:
            assert n == 4_000_000
        row = {"humans": n, "scratch_bytes_default": int(lib.snp_large_scratch_bytes(n, n, L.SNP_F64))}
        crowd = LargeCrowd(MODEL, S, G, dtype=torch.float64, unit_capacity="auto")
        crowd.step(DT, n_substeps=1)  # "auto" settles on its capacity
        crowd.step(DT, n_substeps=1)
        (row["ms_auto"],) = alternated([crowd], args.substeps, max(5, args.reps // 2), 1)
        st = crowd.unit_stats()
        row.update(capacity=st["capacity"], units_listed=st["max_listed"], fallback_units=st["fallback_units"], scratch_bytes_auto=crowd.scratch.numel())
        del crowd
        torch.cuda.empty_cache()
        if row["scratch_bytes_default"] < 0.6 * total:
            crowd = LargeCrowd(MODEL, S, G, dtype=torch.float64)
            (row["ms_default"],) = alternated([crowd], args.substeps, max(5, args.reps // 2), 1)
            del crowd
            torch.cuda.empty_cache()
        else:
            row["ms_default"] = "does not fit"
        result[f"{n}_f64"] = row
        print(json.dumps({f"{n}_f64": row}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
