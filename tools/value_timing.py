"""What CADRL's action choice costs with the value network fused into the lookahead (snp_value_lookahead, predict_from) against the
hand-off it replaces (lookahead_from writes the rotated rows, the same nn.Sequential reads them back in PyTorch, then min / combine /
argmax in torch), with CADRL's default widths (13, 150, 100, 100, 1), gamma 0.9, 81 actions, constant-velocity `next`:

* 4096 envs x 25 humans in fp64 and fp32 (CrowdEngine, one CTA per env and action range), and
* 16 envs x 4096 humans in fp64 (TiledCrowdEngine; the humans split over CTAs in chunks of 256).

Per shape and path: the CUDA-event time of one decision (median, min, max of --reps after --warmup); for the fused path also the
device time of k_value alone (torch.profiler, a separate pass), the network's FLOP/s from shape-derived MACs (rows x sum in*out, two
FLOP each) over that kernel time, and its share of the FP32 FFMA peak that snp_measure_pipe_peak measures in the same run (the path is
FFMA; DESIGN 4.7).  The unfused path runs the network over --chunk envs at a time so its activations fit.  Both paths' choices are
compared.  Prints one JSON line with the GPU's name and power limit, read in the same run (--out: also into a file).

    python tools/value_timing.py [--reps 20] [--warmup 3] [--chunk 256] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from large_lookahead_timing import actions, envs  # noqa: E402
from large_robot_timing import gpu_info, time_ms  # noqa: E402
from social_navigation_pyenvs_b200 import CrowdEngine, TiledCrowdEngine, _lib as L  # noqa: E402

DT, GAMMA, MODEL = 0.25, 0.9, "hsfm_farina"
WIDTHS = (13, 150, 100, 100, 1)
SHAPES = ((4096, 25, torch.float64), (4096, 25, torch.float32), (16, 4096, torch.float64))


def network():
    torch.manual_seed(0)
    layers = []
    for i in range(len(WIDTHS) - 1):
        layers.append(torch.nn.Linear(WIDTHS[i], WIDTHS[i + 1]))
        if i + 2 < len(WIDTHS):
            layers.append(torch.nn.ReLU())
    return torch.nn.Sequential(*layers).cuda()


def unfused(eng, net, nxt, chunk):
    rot, rew = eng.lookahead_from(nxt, DT, yaw_from_next=True)
    with torch.no_grad():
        m = torch.cat([net(rot[i:i + chunk].float()).squeeze(-1).amin(-1) for i in range(0, eng.E, chunk)])
    values = rew + GAMMA ** (DT * eng.robot[L.ROBOT_VD].double())[:, None] * m.double()
    return values.argmax(1), values


def kernel_ms(fn, reps):
    """Mean device time per call of each kernel launched by fn, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type is not None and "CUDA" in str(ev.device_type) and ev.count:
            out[ev.key] = getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 1e3 / reps
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--chunk", type=int, default=256)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("value_timing needs a CUDA device")
    name, power = gpu_info()
    lib = L.lib()
    peak = ctypes.c_double()
    L.check(lib.snp_measure_pipe_peak(0, ctypes.byref(peak)))  # TFLOP/s of a register-resident FP32 FMA loop on every SM
    net = network()
    macs_per_row = sum(WIDTHS[i] * WIDTHS[i + 1] for i in range(len(WIDTHS) - 1))
    res = {"gpu": name, "power_limit": power, "fp32_ffma_peak_tflops_measured": peak.value, "widths": WIDTHS, "actions": 81,
           "unfused_chunk_envs": args.chunk, "reps": args.reps, "shapes": []}
    for E, N, dtype in SHAPES:
        S, G, R = envs(E, N)
        cls = CrowdEngine if N <= 512 else TiledCrowdEngine
        eng = cls.from_reference_arrays(MODEL, S, G, consider_robot=False, all_params_equal=True, robot=R, dtype=dtype)
        eng.set_action_space(actions())
        eng.set_value_network(net, GAMMA)
        nxt = eng.constant_velocity_next(DT).clone()
        fused = lambda: eng.predict_from(nxt, DT, yaw_from_next=True)
        best_f, values_f, _ = (t.clone() for t in fused())
        best_u, values_u = unfused(eng, net, nxt, args.chunk)
        fused_ms = time_ms(fused, args.reps, args.warmup)
        unfused_ms = time_ms(lambda: unfused(eng, net, nxt, args.chunk), args.reps, args.warmup)
        kern = kernel_ms(fused, args.reps)
        k_value = sum(v for k, v in kern.items() if "k_value" in k and "fold" not in k)
        k_fold = sum(v for k, v in kern.items() if "k_value_fold" in k)
        rows = E * 81 * N
        flops = 2.0 * rows * macs_per_row
        res["shapes"].append({
            "E": E, "N": N, "dtype": str(dtype).replace("torch.", ""), "rows": rows, "macs_per_row": macs_per_row,
            "fused_ms": fused_ms, "unfused_ms": unfused_ms, "speedup": unfused_ms[0] / fused_ms[0],
            "k_value_ms": k_value, "k_value_fold_ms": k_fold,
            "k_value_tflops": flops / (k_value * 1e-3) / 1e12 if k_value else None,
            "share_of_fp32_ffma_peak": flops / (k_value * 1e-3) / 1e12 / peak.value if k_value else None,
            "bound": "FP32 FFMA (compute)",
            "choices_equal": float((best_f == best_u).double().mean()),
            "max_abs_value_diff": float((values_f - values_u).abs().max()),
        })
        del eng
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
