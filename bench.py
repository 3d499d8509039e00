#!/usr/bin/env python
"""bench.py -- HSFM agent-steps/s of the fused crowd step on B200, next to the reference algorithm on the host CPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dtype f64|f32] [--workload NAME] [--dump-outputs DIR]

One "step" = one SocialNavGym.step over the whole batch: swept collision / goal / reward checks, then 20 fused
(robot.step + update_humans) sub-steps at dt = 0.0125 (social_gym/social_nav_gym.py:227-250) -- ONE kernel launch.
agent-steps per step = envs x humans x 20.

Default workload = BASELINE.json configs[2]: 4096 envs x 25 humans, HSFM (hsfm_farina), static obstacles (3 zero-speed
humans, reference CCSO style) + the 3 wall polygons of config_example.py, robot visible, collision checks on.
Multi-GPU (torchrun): every rank steps its own 4096 envs (no data-path collective) -> weak scaling.
"""
import argparse
import json
import os
import tempfile
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DT, SUBSTEPS = 0.0125, 20
SETTLE_STEPS = 100
METRIC = "HSFM agent-steps/sec (envs x humans x steps)"
WORKLOADS = {
    # name: (model, E, N, walls, consider_robot)
    "4096x25_hsfm_ccso_walls_robot": ("hsfm_farina", 4096, 25, True, True),
    "4096x25_hsfm_ccso_robot": ("hsfm_farina", 4096, 25, False, True),
    "4096x5_sfm_helbing_cc": ("sfm_helbing", 4096, 5, False, False),
    # the same crowd at a batch size that fills the GPU's warp slots (4096 x 5 occupies 683 of 2368 resident warps: latency-bound)
    "32768x5_sfm_helbing_cc": ("sfm_helbing", 32768, 5, False, False),
    # BASELINE configs[4]: ONE crowd of 65536 humans, sharded by agent across the GPUs (strong scaling, all-gather per sub-step)
    "65536_hsfm_single_crowd": ("hsfm_farina", 1, 65536, False, False),
    # BASELINE configs[3]: 4096 envs x 360-ray laser over 25 humans + 14 wall segments (metric: rays/s)
    "laser_4096x360": ("hsfm_farina", 4096, 25, True, True),
    # SURVEY 8(f)-3: the value-network policies' one-step lookahead for 4096 envs x 81 actions x 25 humans (metric: rotated rows/s)
    "lookahead_4096x81x25": ("hsfm_farina", 4096, 25, True, False),
}


def build_inputs(workload, seed0):
    from social_navigation_pyenvs_b200 import scenarios
    model, E, N, with_walls, robot_visible = WORKLOADS[workload]
    E = int(os.environ.get("SNP_BENCH_ENVS", E))  # tuning experiments only (wave quantisation); the reported workloads use the table
    # per-box scratch (several ranks / several bench runs on one box share it); NOT under gpurun_out/, whose size is capped
    cache = os.path.join(tempfile.gettempdir(), "snp_b200_scenarios", f"scenario_{workload}_{E}_{seed0}.npz")
    if os.path.exists(cache):
        z = np.load(cache)
        sc = dict(states=z["states"], goals=z["goals"], robot=z["robot"])
    else:
        sc = scenarios.ccso_synthetic(E, N, seed0) if "ccso" in workload else scenarios.circular_crossing(E, N, seed0)
        try:
            os.makedirs(os.path.dirname(cache), exist_ok=True)
            tmp = f"{cache}.{os.getpid()}.npz"   # ranks of one job race for the same file: write aside, publish atomically
            np.savez(tmp, **sc)
            os.replace(tmp, cache)
        except OSError:
            pass
    walls = scenarios.pack_walls(scenarios.EXAMPLE_WALLS) if with_walls else None
    states = np.concatenate([sc["states"], sc["robot"][:, None]], 1) if robot_visible else sc["states"]
    safety = np.zeros(states.shape[:2])
    return dict(model=model, E=E, N=N, walls=walls, robot_visible=robot_visible, states=states, goals=sc["goals"],
                robot=sc["robot"], safety=safety)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: the arrays the timed path returned in its last step, one out_dir/<name>.npy each -- float32 data as float32,
    everything else (float64 data, int32 flags and indices) as float64 -- so that two builds can be compared output for output."""
    import torch
    host = {}
    for name, a in arrays.items():
        a = a.cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
        host[name] = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def algorithmic_cost(inp):
    """Per agent-sub-step figures of SURVEY.md 8(d): bytes for ONE HBM round trip of the state a launch touches
    (divided by the fused sub-steps outside), flops F = P*f_pair + f_self + sum_walls(20*S_w + 35), SFU ops."""
    model, N = inp["model"], inp["N"]
    headed = model.startswith("hsfm")
    soc = 1 if "guo" in model else (2 if "moussaid" in model else 0)
    f_pair = (31, 35, 110)[soc]
    P = N - 1 + (1 if inp["robot_visible"] else 0)
    segs = [] if inp["walls"] is None else [int((~np.isnan(w[:, 0, 0])).sum()) for w in inp["walls"]]
    flops = P * f_pair + (150 if headed else 50) + sum(20 * s + 35 for s in segs)
    sfu = (3, 4, 9)[soc] * P + (8 if headed else 4) + sum(s + 3 for s in segs)
    words = 19 if headed else 13  # SURVEY 8(d): HSFM reads 11 + writes 8 words, SFM reads 9 + writes 4
    return dict(flops=flops, sfu=sfu, words=words)


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region, polled through NVML every few ms (the same counters as the
    nvidia-smi line of B200_PROFILING.md: clocks.sm, clocks.max.sm, clocks_event_reasons.*)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.sm, self.bits, self.max_mhz, self.stop, self.thread = index, [], 0, None, False, None

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)

            period = float(os.environ.get("SNP_CLOCK_POLL_MS", "4")) * 1e-3

            def poll():
                while not self.stop:
                    self.sm.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                    self.bits |= pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                    time.sleep(period)
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
        except Exception:
            self.thread = None
        return self

    def __exit__(self, *a):
        self.stop = True
        if self.thread:
            self.thread.join(timeout=1)

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(self.sm), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for b, n in self.REASONS.items() if self.bits & b), "samples": len(self.sm)}


def measured_traffic(args):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE k_step launch from the committed `ncu --set full` capture of this
    exact workload / dtype (profiles/traffic.json), or None."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[f"{args.workload}:{args.dtype}"]
    except (OSError, KeyError, ValueError):
        return None


def issue_model(key, clocks, measured_ms):
    """Pipe / issue bound of the dominant kernel: warp instructions of ONE launch from the committed ncu capture of this workload
    (profiles/issue_model.json, written by tools/issue_cost.py), costed with the pipe figures tools/pipe_microbench.cu measured on
    B200 (profiles/r02_pipe_microbench.txt): DFMA 3.0 cycles of its SMSP's FP64 pipe, DMUL / DADD / DSETP 2.06, FMA-pipe instructions
    on the same dispatch port, ALU-pipe instructions overlapping at 2 cycles each; bound = max(port, ALU, issue slots), at the SM
    clock sampled during the timed region."""
    try:
        m = json.load(open(os.path.join(ROOT, "profiles", "issue_model.json")))[key]
        mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz")
        bound_ms = m["issue_cycles_per_smsp"] / (mhz * 1e3)
        return {"bound_ms": bound_ms, "frac": bound_ms / measured_ms, "fp64_warp_instructions": m["fp64_warp_instructions"],
                "other_warp_instructions": m["other_warp_instructions"], "fp64_issue_cycles": m["fp64_issue_cycles"],
                "port_cycles_per_smsp": m.get("port_cycles_per_smsp"), "alu_cycles_per_smsp": m.get("alu_cycles_per_smsp"),
                "issue_slots_per_smsp": m.get("issue_slots_per_smsp"), "sm_mhz": mhz,
                "source": "profiles/issue_model.json (" + m["source"] + ")"}
    except (OSError, KeyError, ValueError, TypeError):
        return None


def oracle_rate(inp, n_envs, threads, substeps, repeats=1):
    """The reference's algorithm on the host: C restatement (oracle/snp_oracle.c, serial semantics), OpenMP over envs."""
    import oracle
    from oracle import OracleConfig
    cfg = OracleConfig(oracle.type_code(inp["model"]), inp["robot_visible"], True, False)
    N = inp["N"]
    S, G = inp["states"][:n_envs], inp["goals"][:n_envs]
    params = np.tile(oracle.default_params(inp["model"]), (n_envs, N, 1))
    D = np.zeros((n_envs, N, 2))
    rv = np.tile([0.0, 1.0], (n_envs, 1))
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        oracle.update_humans(cfg, S, G, inp["walls"], params, inp["safety"][:n_envs], D, DT, substeps,
                             robot_vel=rv if inp["robot_visible"] else None, n_threads=threads)
        best = min(best, time.perf_counter() - t0)
    return n_envs * N * substeps / best, best


def workload_config(workload, inp):
    """The `config` object of BOTH arms (same keys, same values: the driver compares them)."""
    return {"workload": workload, "envs_per_gpu": inp["E"], "humans": inp["N"], "motion_model": inp["model"], "substeps_per_step": SUBSTEPS,
            "dt": DT, "walls": 0 if inp["walls"] is None else int(inp["walls"].shape[0]), "robot_visible": inp["robot_visible"],
            "checks": "swept collision/goal/reward + per-sub-step touch", "l2": "256 MiB flush write between timed steps",
            "timing": "sum of per-step CUDA-event pairs on the launch stream, max over ranks"}


def pin_host_threads(local_rank, world):
    """Keep this rank's host threads (and the pinned buffers they first touch) on the cores next to its GPU: the GPU's NUMA-local
    cpulist from sysfs intersected with the allowed set, split evenly between the ranks that share it.  Best effort; returns a note."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[local_rank]) if vis and vis.split(",")[local_rank].isdigit() else local_rank
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(phys)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        path = f"/sys/bus/pci/devices/{bus[-12:].lower()}/local_cpulist"
        local = set()
        for part in open(path).read().strip().split(","):
            lo, _, hi = part.partition("-")
            local.update(range(int(lo), int(hi or lo) + 1))
        allowed = sorted(os.sched_getaffinity(0))
        near = [c for c in allowed if c in local] or allowed
        if world > 1:  # ranks whose GPUs share this cpulist split it (contiguous slices, at least 2 cores each)
            share = max(2, len(near) // world)
            lo = (local_rank * share) % max(1, len(near) - share + 1)
            near = near[lo:lo + share]
        os.sched_setaffinity(0, near)
        return f"rank {local_rank}: {len(near)} cores {near[0]}-{near[-1]} (GPU-local cpulist {'hit' if local & set(allowed) else 'outside the allowed set'})"
    except Exception as exc:  # no NVML / sysfs entry: leave the affinity alone
        return f"unchanged ({type(exc).__name__})"


def host_threads():
    return len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)


def reference_pool(inp, n_procs):
    """The LIVE reference (staged under oracle/_ref by oracle/build.py, or /root/reference): n_procs resident processes, one env
    each, serial MotionModelManager.update_humans path (parallelize_humans=False) -- BASELINE.md section 4.  None when not staged."""
    from oracle import reference
    if not reference.available() or inp["E"] == 1:
        return None
    from social_navigation_pyenvs_b200 import scenarios
    walls = scenarios.EXAMPLE_WALLS if inp["walls"] is not None else None
    return reference.ReferencePool(n_procs, inp["model"], inp["states"], inp["goals"], walls, inp["robot"], inp["robot_visible"], DT)


def reference_baseline(inp, seconds=10.0):
    """cpu_baseline of the GPU arm: ~`seconds` of the live reference on all host cores (call BEFORE CUDA is initialised: the pool forks)."""
    threads = host_threads()
    pool = reference_pool(inp, threads)
    if pool is None:
        return None
    try:
        pool.step(SUBSTEPS)
        spent, reps = 0.0, 0
        while spent < seconds:
            t, _ = pool.step(SUBSTEPS)
            spent += t; reps += 1
    finally:
        pool.close()
    return {"value": threads * inp["N"] * SUBSTEPS * reps / spent, "unit": "agent-steps/s", "cores": threads, "kind": "reference",
            "sample": f"{reps} gym steps x ({threads} of {inp['E']} envs, one per process, {SUBSTEPS} sub-steps each) of the live reference: "
                      f"SocialNavSim + MotionModelManager.update_humans, serial Python/NumPy path (motion_model_manager.py:354-373)"}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores -- the live Python reference
    (one env per process on every core; a step = one gym step = 20 sub-steps of those envs), or, where it is not staged, the
    oracle port with OpenMP over envs.  Rank 0 only."""
    if rank != 0:
        return
    inp = build_inputs(args.workload, 2000)
    threads = host_threads()
    pool = reference_pool(inp, threads)
    if pool is not None:
        try:
            for _ in range(args.warmup):
                pool.step(SUBSTEPS)
            times = [pool.step(SUBSTEPS)[0] for _ in range(args.steps)]
        finally:
            pool.close()
        total = sum(times)
        value = threads * inp["N"] * SUBSTEPS * args.steps / total
        sample = (f"{threads} of {inp['E']} envs per step, one per process on {threads} host cores, {SUBSTEPS} sub-steps each: the live reference "
                  f"(SocialNavSim + MotionModelManager.update_humans, serial Python/NumPy path, motion_model_manager.py:354-373)")
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "agent-steps/s", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(args.workload, inp),
                "notes": "host wall clock per step (no GPU); the reference arm times the motion update only, without the checks",
                "cpu_baseline": {"value": value, "unit": "agent-steps/s", "cores": threads, "kind": "reference", "sample": sample},
                "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return
    n_envs = min(inp["E"], max(threads * 4, 128))
    for _ in range(args.warmup):
        oracle_rate(inp, n_envs, threads, 2)
    times = []
    for _ in range(args.steps):
        _, t = oracle_rate(inp, n_envs, threads, SUBSTEPS)
        times.append(t)
    total = sum(times)
    value = n_envs * inp["N"] * SUBSTEPS * args.steps / total
    sample = f"{n_envs} of {inp['E']} envs x {SUBSTEPS} sub-steps per step, C restatement of the serial Python/NumPy path, OpenMP over envs"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "agent-steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.workload, inp),
            "notes": "host wall clock per step (no GPU); live reference not staged, C port of its serial path timed instead",
            "cpu_baseline": {"value": value, "unit": "agent-steps/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_large_crowd(args, rank, world, local_rank):
    """Config 5: one 65536-human HSFM crowd (256 x 256 jittered grid, SURVEY.md 8(d)); a step = ONE sub-step = one tiled
    all-pairs launch per rank + one all-gather of the [5, N] entity view.  Total work is fixed -> strong scaling."""
    import ctypes
    import torch
    import torch.distributed as dist
    from social_navigation_pyenvs_b200 import scenarios, _lib
    from social_navigation_pyenvs_b200.large import LargeCrowd
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = _lib.lib()
    tdtype = torch.float64 if args.dtype == "f64" else torch.float32
    sc = scenarios.jittered_grid_crowd(256, pitch=2.0, jitter=0.5, seed=0)
    n = sc["states"].shape[1]
    order = os.environ.get("SNP_LARGE_ORDER", "patch")
    if order == "patch":  # number the humans patch by patch: compact tiles for the exact far-tile culling (scenarios.spatial_order)
        perm = scenarios.spatial_order(sc["states"][0, :, 0:2])
        sc = dict(states=np.ascontiguousarray(sc["states"][:, perm]), goals=np.ascontiguousarray(sc["goals"][:, perm]))
    crowd = LargeCrowd("hsfm_farina", sc["states"][0], sc["goals"][0], dtype=tdtype, rank=rank, world=world,
                       exchange=os.environ.get("SNP_EXCHANGE", "auto"))
    steps = args.steps
    for _ in range(args.warmup):
        crowd.step(DT, 1)
    crowd.check_peers()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    stream = torch.cuda.current_stream()
    lib.snp_launch_count(1)
    with ClockSampler(local_rank) as clocks:
        for s in range(steps):
            flush.fill_(s & 0xFF)
            ev[s][0].record(stream)
            crowd.step(DT, 1)
            ev[s][1].record(stream)
        torch.cuda.synchronize()
    launches = int(lib.snp_launch_count(0))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"dyn": crowd.eng.dyn, "goal_idx": crowd.eng.goal_idx})
    from social_navigation_pyenvs_b200.parallel import max_over_ranks
    total_ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in ev), "cuda", world)
    # the same steps with the exact far-tile culling switched off: every ordered pair is evaluated -> the all-pairs roofline
    crowd.culling = False
    crowd.step(DT, 1)
    ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(max(3, steps // 3))]
    for a_, b_ in ev2:
        flush.fill_(1)
        a_.record(stream)
        crowd.step(DT, 1)
        b_.record(stream)
    torch.cuda.synchronize()
    allpairs_ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in ev2), "cuda", world) / len(ev2)
    crowd.culling = True
    # end to end: host rows in, host rows out around one sub-step of the whole crowd (public API of LargeCrowd)
    tmpl = sc["states"][0][crowd.offset:crowd.offset + crowd.n_local]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        crowd.eng.load_rows(tmpl[None])
        crowd._publish()
        crowd.step(DT, 1)
        crowd.local_rows(tmpl)
    e2e_s = max_over_ranks(time.perf_counter() - t0, "cuda", world)
    if rank == 0:
        pipe = ctypes.c_double()
        _lib.check(lib.snp_measure_pipe_peak(1 if args.dtype == "f64" else 0, ctypes.byref(pipe)))
        flops = n * ((n - 1) * 31 + 150)  # SURVEY 8(d): 65535 ordered pairs x 31 + 150 per agent-step
        per_s = allpairs_ms * 1e-3
        ach = flops / per_s / 1e12
        line = {"metric": METRIC, "value": n * steps / (total_ms * 1e-3), "unit": "agent-steps/s", "n_gpus": world, "steps": steps,
                "warmup": args.warmup, "ms_per_step": total_ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": args.dtype, "data": "synthetic",
                "config": {"workload": args.workload, "humans": n, "motion_model": "hsfm_farina", "substeps_per_step": 1, "dt": DT,
                           "sharding": f"by agent over {world} GPU(s); entity view [5,N] exchanged per sub-step via " +
                                       ("peer (NVLink) stores fused into the producer kernel + barrier" if crowd.exchange == "p2p" else "NCCL all-gather"),
                           "culling": "exact far-tile culling on for `value` (tiles beyond the exp-underflow distance contribute exactly 0); "
                                      "roofline measured with culling off (every ordered pair evaluated)",
                           "ms_per_step_all_pairs": allpairs_ms,
                           "agent_order": "patch by patch (scenarios.spatial_order of the initial positions: runs of 256 humans cover ~31 m x 31 m)"
                                          if order == "patch" else "row by row of the 256 x 256 grid (runs of 256 humans cover 510 m x 1 m)",
                           "l2": "256 MiB flush write between timed steps"},
                "clocks": clocks.summary(), "gpu_launches": launches,
                "e2e": {"value": n * reps / e2e_s, "unit": "agent-steps/s", "h2d_bytes_per_step": int(tmpl.size * 8), "d2h_bytes_per_step": int(tmpl.size * 8),
                        "api": "LargeCrowd: load_rows (H2D) + step + local_rows (D2H)", "steps": reps},
                "roofline": {"bound": "fp64" if args.dtype == "f64" else "fp32", "achieved": ach * world / world, "peak": pipe.value * world, "unit": "TFLOP/s",
                             "frac": ach / (pipe.value * world), "traffic": None, "kernel": "snp::k_large_pairs (tiled all-pairs, culling off)",
                             "flops_per_agent_substep": (n - 1) * 31 + 150,
                             "peak_source": "measured in this run on rank 0 (snp_measure_pipe_peak) x n_gpus"}}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def large_crowd_probe(tdtype, rank, world, substeps_per_call=10, calls=3):
    """BASELINE configs[4] beside the default line, at every N: ONE crowd of 65536 HSFM humans sharded by agent over the N GPUs,
    the sub-step loop inside one C call (snp_large_run_p2p: peer stores of entries + tile boxes fused into the producer, a
    single-warp barrier kernel between sub-steps).  Returns ms per sub-step (device time, max over ranks), the exchange in use
    and whether this rank's slice equals the single-GPU result bit for bit."""
    import torch
    from social_navigation_pyenvs_b200 import scenarios
    from social_navigation_pyenvs_b200.large import LargeCrowd
    from social_navigation_pyenvs_b200.parallel import max_over_ranks
    sc = scenarios.jittered_grid_crowd(256, pitch=2.0, jitter=0.5, seed=0)
    perm = scenarios.spatial_order(sc["states"][0, :, 0:2])
    if world > 1 and os.environ.get("SNP_LARGE_DEAL", "1") == "1":
        # load balance: the 128-human tiles (compact patches) are dealt to the ranks round-robin, so every rank owns patches from
        # all over the crowd instead of one block of strips (an interior block has ~25 % more near neighbours than a corner one).
        # The numbering is the caller's; no force depends on it.
        perm = scenarios.deal_tiles(perm, world)
    S, G = np.ascontiguousarray(sc["states"][0, perm]), np.ascontiguousarray(sc["goals"][0, perm])
    n = S.shape[0]
    crowd = LargeCrowd("hsfm_farina", S, G, dtype=tdtype, rank=rank, world=world, exchange=os.environ.get("SNP_EXCHANGE", "auto"))
    stream = torch.cuda.current_stream()

    def timed(k, reps):
        crowd.step(DT, k)  # warm-up call
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a_, b_ in ev:
            a_.record(stream)
            crowd.step(DT, k)
            b_.record(stream)
        torch.cuda.synchronize()
        return max_over_ranks(sum(a_.elapsed_time(b_) for a_, b_ in ev), "cuda", world) / (reps * k)

    # bit-equality first (from the initial state): 4 sub-steps sharded vs the whole crowd on this GPU alone
    crowd.step(DT, 4)
    mine = crowd.local_rows(S[crowd.offset:crowd.offset + crowd.n_local])
    equal = True
    if world > 1:
        single = LargeCrowd("hsfm_farina", S, G, dtype=tdtype, rank=0, world=1)
        single.step(DT, 4)
        equal = bool(np.array_equal(mine, single.local_rows(S)[crowd.offset:crowd.offset + crowd.n_local]))
        del single
        equal = max_over_ranks(0.0 if equal else 1.0, "cuda", world) == 0.0
    culled = timed(substeps_per_call, calls)
    crowd.culling = False
    allpairs = timed(2, 1)
    crowd.culling = True
    crowd.check_peers()
    return {"workload": "65536_hsfm_single_crowd", "humans": n, "n_gpus": world, "scaling": "strong", "dtype": "f64" if tdtype == torch.float64 else "f32",
            "ms_per_substep": culled, "agent_steps_per_s": n / (culled * 1e-3), "ms_per_substep_all_pairs": allpairs,
            "exchange": {"p2p": "peer (NVLink) stores of entries + tile boxes fused into the finish kernel, device-side barrier kernel, "
                                "sub-step loop in one C call (snp_large_run_p2p)",
                         "fused": "single GPU: sub-step loop in one C call (snp_large_run_p2p), no exchange",
                         "nccl": "NCCL all-gather of the [5, N] view per sub-step"}[crowd.exchange],
            "pair_phase": "k_large_cull lists the (i-block, 128-entity chunk) units in reach; persistent CTAs with one queue per SM work the list off",
            "substeps_per_call": substeps_per_call, "bit_equal_to_single_gpu": equal, "timing": "CUDA events around each call, max over ranks",
            "agent_order": "patch by patch (scenarios.spatial_order)" + (", 128-human tiles dealt round-robin to the ranks" if world > 1 and os.environ.get("SNP_LARGE_DEAL", "1") == "1" else "")}


def run_laser(args, rank, world, local_rank):
    """Config 4: LaserSensor.get_laser_measurements for 4096 sensors x 360 rays (range 2 pi, max 10 m) over the 25 humans and the
    3 wall polygons (14 segments) of workload 3b; a step = one scan of every env = one launch.  Env-sharded (weak scaling)."""
    import ctypes
    inp = build_inputs("4096x25_hsfm_ccso_walls_robot", 2000 + rank * 4096)
    import torch
    import torch.distributed as dist
    from social_navigation_pyenvs_b200 import CrowdEngine, _lib, sensors
    from social_navigation_pyenvs_b200.parallel import max_over_ranks
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = _lib.lib()
    tdtype = torch.float64 if args.dtype == "f64" else torch.float32
    E, N, samples = inp["E"], inp["N"], 360
    eng = CrowdEngine.from_reference_arrays(inp["model"], inp["states"], inp["goals"], walls=inp["walls"], safety=inp["safety"],
                                            consider_robot=True, all_params_equal=True, dtype=tdtype)
    pose = torch.stack([eng.robot[_lib.ROBOT_PX], eng.robot[_lib.ROBOT_PY], torch.full((E,), float(np.pi / 2), dtype=tdtype, device="cuda")])
    pose = pose.contiguous()
    scanner = sensors.EngineScanner(eng, 2 * np.pi, samples, 10.0, robot_radius=0.3)
    for _ in range(args.warmup):
        scanner.scan(pose)
    torch.cuda.synchronize()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    if world > 1:
        dist.barrier()
    lib.snp_launch_count(1)
    with ClockSampler(local_rank) as clocks:
        for s in range(args.steps):
            flush.fill_(s & 0xFF)
            ev[s][0].record(stream)
            ranges, hits = scanner.scan(pose)
            ev[s][1].record(stream)
        torch.cuda.synchronize()
    launches = int(lib.snp_launch_count(0))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"ranges": ranges, "hits": hits})
    total_ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in ev), "cuda", world)
    # end to end with host arrays through the reference-shaped call (humans [E,N,3], walls, pose [E,3] -> ranges, hits)
    humans = inp["states"][:, :N][:, :, [0, 1, 8]].copy()
    pose_h = np.concatenate([inp["robot"][:, 0:2], np.full((E, 1), np.pi / 2)], 1)
    sensors.scan_batch(humans, inp["walls"], pose_h, 2 * np.pi, samples, 10.0, 0.3, dtype="float64" if args.dtype == "f64" else "float32")
    t0 = time.perf_counter()
    for _ in range(5):
        sensors.scan_batch(humans, inp["walls"], pose_h, 2 * np.pi, samples, 10.0, 0.3, dtype="float64" if args.dtype == "f64" else "float32")
    batch_s = max_over_ranks(time.perf_counter() - t0, "cuda", world) / 5
    # end to end on the RESIDENT crowd (what a robot with a laser does every step): pinned pose in, ranges + hit indices written by
    # the kernel straight into pinned host buffers, sync
    pose_pin = pose.cpu().pin_memory()
    ranges_pin = torch.empty((E, samples), dtype=tdtype).pin_memory()
    hits_pin = torch.empty((E, samples), dtype=torch.int32).pin_memory()
    reps, ts = 100, []
    for it in range(5 + reps):
        t0 = time.perf_counter()
        scanner.scan_host(pose_pin, ranges_pin, hits_pin)
        if it >= 5:
            ts.append(time.perf_counter() - t0)
    assert torch.equal(ranges_pin, scanner.scan(pose)[0].cpu())
    e2e_s = max_over_ranks(statistics.median(ts), "cuda", world) * reps
    if rank == 0:
        pipe = ctypes.c_double()
        _lib.check(lib.snp_measure_pipe_peak(1 if args.dtype == "f64" else 0, ctypes.byref(pipe)))
        nseg = int((~np.isnan(inp["walls"][:, :, 0, 0])).sum())
        flops_per_ray = 12 * N + 25 * nseg  # SURVEY 8(d)
        per_s = total_ms / args.steps * 1e-3
        ach = E * samples * flops_per_ray / per_s / 1e12
        w = 8 if args.dtype == "f64" else 4
        bytes_per_launch = E * ((3 * N + 3) * w + samples * (w + 4)) + 4 * nseg * w
        line = {"metric": "laser rays/sec (envs x rays)", "value": world * E * samples * args.steps / (total_ms * 1e-3), "unit": "rays/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
                "config": {"workload": args.workload, "envs_per_gpu": E, "rays": samples, "humans": N, "wall_segments": nseg,
                           "l2": "256 MiB flush write between timed steps"},
                "clocks": clocks.summary(), "gpu_launches": launches,
                "e2e": {"value": world * E * samples * reps / e2e_s, "unit": "rays/s", "h2d_bytes_per_step": int(pose_pin.numel() * pose_pin.element_size()),
                        "d2h_bytes_per_step": int(ranges_pin.numel() * ranges_pin.element_size() + hits_pin.numel() * 4),
                        "api": "EngineScanner.scan_host on the resident crowd: pinned pose in, ranges + hits written by the kernel into pinned host buffers, sync",
                        "steps": reps, "statistic": "median call, max over ranks",
                        "scan_batch_host_arrays_rays_per_s": world * E * samples / batch_s},
                "roofline": {"bound": "fp64" if args.dtype == "f64" else "fp32", "achieved": ach, "peak": pipe.value, "unit": "TFLOP/s",
                             "frac": ach / pipe.value, "traffic": measured_traffic(args), "kernel": "snp::k_laser_rays", "flops_per_ray": flops_per_ray,
                             "hbm": {"achieved_gbs": bytes_per_launch / per_s / 1e9, "bytes_per_ray": bytes_per_launch / (E * samples)}}}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_lookahead(args, rank, world, local_rank):
    """SURVEY 8(f)-3: what CADRL.predict computes per decision (crowd_nav/policy/cadrl.py:235-262) for every env at once: peek of the
    humans at dt = 0.25 (1 launch of k_step into a side buffer) + rewards and agent-centric states of the 81 actions (1 launch of
    k_lookahead, 862 MB of output in fp64 -> HBM-write bound).  A step = both launches.  Env-sharded (weak scaling)."""
    inp = build_inputs("4096x25_hsfm_ccso_walls_robot", 2000 + rank * 4096)
    import torch
    import torch.distributed as dist
    from social_navigation_pyenvs_b200 import CrowdEngine, _lib
    from social_navigation_pyenvs_b200.parallel import max_over_ranks
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = _lib.lib()
    tdtype = torch.float64 if args.dtype == "f64" else torch.float32
    E, N = inp["E"], inp["N"]
    robot = inp["robot"].copy()
    robot[:, 12] = 1.0
    eng = CrowdEngine.from_reference_arrays(inp["model"], inp["states"][:, :N], inp["goals"], walls=inp["walls"], safety=inp["safety"][:, :N],
                                            consider_robot=False, all_params_equal=True, dtype=tdtype, robot=robot)
    speeds = [(np.exp((i + 1) / 5) - 1) / (np.e - 1) for i in range(5)]  # cadrl.py build_action_space, holonomic, v_pref = 1
    rots = np.linspace(0, 2 * np.pi, 16, endpoint=False)
    actions = np.array([[0.0, 0.0]] + [[sp * np.cos(r), sp * np.sin(r)] for r in rots for sp in speeds])
    eng.set_action_space(actions)
    A, OW = actions.shape[0], 13
    bulk = os.environ.get("SNP_LOOKAHEAD_STORE", "bulk") == "bulk"
    for _ in range(args.warmup):
        eng.lookahead(0.25, bulk_store=bulk)
    torch.cuda.synchronize()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    if world > 1:
        dist.barrier()
    lib.snp_launch_count(1)
    with ClockSampler(local_rank) as clocks:
        for s in range(args.steps):
            flush.fill_(s & 0xFF)
            ev[s][0].record(stream)
            nxt = eng.peek(0.25)
            ev[s][1].record(stream)
            rot, rew = eng.lookahead_from(nxt, 0.25, bulk_store=bulk)
            ev[s][2].record(stream)
        torch.cuda.synchronize()
    launches = int(lib.snp_launch_count(0))
    if args.dump_outputs and rank == 0:
        # the rotated states are 862 MB in fp64: a fixed, seeded sample of 128 envs of them
        envs = np.sort(np.random.default_rng(0).choice(E, min(E, 128), replace=False))
        dump_outputs(args.dump_outputs, {"next": nxt, "rewards": rew, "rotated_envs": envs,
                                         "rotated": rot[torch.from_numpy(envs).to(rot.device)]})
    total_ms = max_over_ranks(sum(e[0].elapsed_time(e[2]) for e in ev), "cuda", world)
    look_ms = sum(e[1].elapsed_time(e[2]) for e in ev) / args.steps
    peek_ms = sum(e[0].elapsed_time(e[1]) for e in ev) / args.steps
    # end to end: the robot's state changes every decision (H2D from pinned memory), the rewards come back (D2H); the rotated
    # states stay on the device, where the value network that consumes them runs (cadrl.py:255-259)
    robot_host = eng.robot.cpu().pin_memory()
    rew_host = torch.empty((E, A), dtype=torch.float64).pin_memory()
    reps = max(10, args.steps // 2)
    for it in range(3 + reps):
        if it == 3:
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
        eng.robot.copy_(robot_host, non_blocking=True)
        _, rew = eng.lookahead(0.25, bulk_store=bulk)
        rew_host.copy_(rew, non_blocking=True)
        torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0, "cuda", world)
    # a write-only reference on the same buffer: what a plain fill of the output achieves on this GPU (the copy peak of
    # MEASURED_PEAKS.json is read + write traffic; a pure write stream tops out lower)
    rot_buf = eng._rotated
    fill_ms = []
    for _ in range(6):
        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        flush.fill_(3)
        a_.record(stream)
        rot_buf.fill_(1.0)
        b_.record(stream)
        torch.cuda.synchronize()
        fill_ms.append(a_.elapsed_time(b_))
    write_only_gbs = rot_buf.numel() * rot_buf.element_size() / (min(fill_ms[1:]) * 1e-3) / 1e9
    if rank == 0:
        w = 8 if args.dtype == "f64" else 4
        rows = E * A * N
        out_bytes = rows * OW * w + E * A * 8
        in_bytes = E * N * 11 * w + E * 6 * w + A * 16
        hbm_peak, hbm_src = 6650.0, "fallback"
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            hbm_peak, hbm_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, copy read+write)"
        ach = (out_bytes + in_bytes) / (look_ms * 1e-3) / 1e9
        line = {"metric": "lookahead rows/sec (envs x actions x humans)", "value": world * rows * args.steps / (total_ms * 1e-3), "unit": "rows/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
                "config": {"workload": args.workload, "envs_per_gpu": E, "actions": A, "humans": N, "values_per_row": OW, "time_step": 0.25,
                           "store": "cp.async.bulk shared->global" if bulk else "per-thread 16-byte stores",
                           "ms_peek": peek_ms, "ms_lookahead": look_ms, "l2": "256 MiB flush write between timed steps; output (862 MB fp64) exceeds L2"},
                "clocks": clocks.summary(), "gpu_launches": launches,
                "e2e": {"value": world * rows * reps / e2e_s, "unit": "rows/s", "h2d_bytes_per_step": int(robot_host.numel() * robot_host.element_size()),
                        "d2h_bytes_per_step": int(rew_host.numel() * 8), "api": "CrowdEngine.lookahead: pinned H2D robot state, peek + lookahead, D2H rewards "
                        "(rotated states stay on the device for the value network)", "steps": reps},
                "roofline": {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": measured_traffic(args),
                             "kernel": "snp::k_lookahead", "bytes_per_row": (out_bytes + in_bytes) / rows, "peak_source": hbm_src,
                             "write_only": {"fill_gbs": write_only_gbs, "frac": ach / write_only_gbs,
                                            "how": "torch fill_ of the same output buffer, best of 5, CUDA events, L2 flushed"}}}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--workload", default="4096x25_hsfm_ccso_walls_robot", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path computed in its last step as DIR/<name>.npy "
                    "(rank 0's share when several GPUs run)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    if args.workload == "65536_hsfm_single_crowd":
        run_large_crowd(args, rank, world, local_rank)
        return
    if args.workload == "laser_4096x360":
        run_laser(args, rank, world, local_rank)
        return
    if args.workload == "lookahead_4096x81x25":
        run_lookahead(args, rank, world, local_rank)
        return
    # host-side scenario generation forks worker processes: do it before CUDA is initialised in this process
    inp = build_inputs(args.workload, 2000 + rank * 4096)  # every rank owns different envs
    E, N = inp["E"], inp["N"]
    # ... and so does the live-reference baseline (rank 0 at N = 1 only): ~10 s of the reference on all host cores
    ref_baseline = reference_baseline(inp) if (not args.no_cpu_baseline and world == 1) else None

    import torch
    import torch.distributed as dist
    from social_navigation_pyenvs_b200 import CrowdEngine, _lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    full_affinity = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    affinity_note = pin_host_threads(local_rank, world)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = _lib.lib()
    tdtype = torch.float64 if args.dtype == "f64" else torch.float32
    def make_engine(dt_):
        return CrowdEngine.from_reference_arrays(inp["model"], inp["states"], inp["goals"], walls=inp["walls"], safety=inp["safety"],
                                                 consider_robot=inp["robot_visible"], all_params_equal=True, dtype=dt_,
                                                 robot=None if inp["robot_visible"] else inp["robot"])

    eng = make_engine(tdtype)
    eng.mapping = int(os.environ.get("SNP_MAPPING", "0"))  # tuning: 1 force warp-packed, 2 force block-packed thread mapping
    action_host = torch.tensor(np.tile([[0.0], [1.0]], (1, E)), dtype=tdtype).pin_memory()  # [2,E] holonomic action
    eng.action.copy_(action_host)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    stream = torch.cuda.current_stream()

    def one_step(e=eng):
        e.step(None, DT, n_substeps=SUBSTEPS, pre_checks=True, post_checks=False, track_touch=True)

    for _ in range(args.warmup):
        one_step()
    torch.cuda.synchronize()
    # extra untimed load so the SM clock has ramped before the timed region starts.  It steps a twin of the engine, so that the
    # state the timed steps start from does not depend on how many ramp steps fit in the ramp time
    twin = make_engine(tdtype)
    twin.mapping = eng.mapping
    twin.action.copy_(action_host)
    t_ramp = time.perf_counter()
    while time.perf_counter() - t_ramp < float(os.environ.get("SNP_BENCH_RAMP_S", "0.25")):
        for _ in range(20):
            one_step(twin)
        torch.cuda.synchronize()
    del twin
    # A fixed number of untimed steps takes the crowd past the opening of the episode: while every human crosses the centre at
    # once (steps ~25-55) a step costs up to 2 % more; from step ~100 on the cost per step is flat.
    for _ in range(SETTLE_STEPS):
        one_step()
    torch.cuda.synchronize()

    # ---- timed region: K steps, each its own CUDA-event pair on the launching stream, L2 flushed between steps ----
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    lib.snp_launch_count(1)
    with ClockSampler(local_rank) as clocks:
        wall0 = time.perf_counter()
        for s in range(args.steps):
            flush.fill_(s & 0xFF)
            ev[s][0].record(stream)
            one_step()
            ev[s][1].record(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - wall0
    launches = int(lib.snp_launch_count(0))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"dyn": eng.dyn, "robot": eng.robot, "goal_idx": eng.goal_idx, "time_now": eng.time_now,
                                         "flags": eng.flags, "checks": eng.checks})
    if world > 1:
        dist.barrier()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = sum(step_ms)
    if os.environ.get("SNP_BENCH_DUMP_STEPS"):  # tuning: per-step times (the crowd's state, hence the branch mix, evolves over the run)
        with open(os.environ["SNP_BENCH_DUMP_STEPS"], "w") as f:
            f.write("\n".join(f"{x:.5f}" for x in step_ms))
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    agent_steps = E * N * SUBSTEPS * args.steps
    value = world * agent_steps / (total_ms * 1e-3)

    # ---- end to end through the public API with HOST buffers: H2D action from pinned memory, launch, D2H of the
    #      observation (px,py,vx,vy of every human), flags, reward/dmin ----
    obs_host = torch.empty((4, E, N), dtype=tdtype).pin_memory()
    flags_host = torch.empty((E,), dtype=torch.int32).pin_memory()
    checks_host = torch.empty((E, 4), dtype=torch.float64).pin_memory()
    e2e_steps = max(100, args.steps)

    def e2e_run(staged):
        """>= 100 calls of the public host-buffer API, each timed on the host clock around the call (it ends with a stream
        synchronisation); the MEDIAN step, max over ranks, is the figure (single stragglers -- another rank's page fault, a
        scheduler tick -- do not decide it)."""
        ts = []
        for it in range(5 + e2e_steps):
            if it == 5 and world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            # ONE C-ABI call with host buffers (snp_gym_step_host): H2D action, fused launch whose store phase writes observation +
            # flags + checks into the pinned buffers (staged: D2H copies after the launch), sync
            eng.step_host(action_host, obs_host, flags_host, checks_host, DT, n_substeps=SUBSTEPS, pre_checks=True, post_checks=False,
                          track_touch=True, staged=staged)
            if it >= 5:
                ts.append(time.perf_counter() - t0)
        med, mean = statistics.median(ts), sum(ts) / len(ts)
        if world > 1:
            t = torch.tensor([med, mean], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            med, mean = float(t[0].item()), float(t[1].item())
        return med, mean

    e2e_med, e2e_mean = e2e_run(staged=False)
    e2e_staged_med, _ = e2e_run(staged=True)
    assert torch.equal(obs_host.view(4, -1), eng.dyn[:4].view(4, -1).cpu()), "host observation differs from the device state"
    e2e_value = world * E * N * SUBSTEPS / e2e_med
    h2d = action_host.numel() * action_host.element_size()
    d2h = sum(x.numel() * x.element_size() for x in (obs_host, flags_host, checks_host))

    # ---- BASELINE configs[4] at this N (all ranks take part): one 65536-human crowd sharded by agent ----
    large = None
    if not os.environ.get("SNP_BENCH_NO_LARGE"):
        del flush
        try:
            large = large_crowd_probe(tdtype, rank, world)
        except Exception as exc:  # keep the headline line even if the side measurement cannot run on this box
            large = {"workload": "65536_hsfm_single_crowd", "error": repr(exc)}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant (only) kernel: k_step ----
    cost = algorithmic_cost(inp)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm_peak, hbm_src = 6650.0, "fallback"
    if os.path.exists(peaks_path):
        hbm_peak, hbm_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured"
    import ctypes
    pipe = ctypes.c_double()
    _lib.check(lib.snp_measure_pipe_peak(1 if args.dtype == "f64" else 0, ctypes.byref(pipe)))
    mufu = ctypes.c_double()
    _lib.check(lib.snp_measure_pipe_peak(2, ctypes.byref(mufu)))
    per_launch_s = (total_ms / args.steps) * 1e-3
    wbytes = 8 if args.dtype == "f64" else 4
    launch_bytes = E * N * cost["words"] * wbytes  # one HBM round trip of the state per launch (k fused sub-steps share it)
    launch_flops = E * N * SUBSTEPS * cost["flops"]
    ach_tflops = launch_flops / per_launch_s / 1e12
    ach_gbs = launch_bytes / per_launch_s / 1e9
    ach_sfu = E * N * SUBSTEPS * cost["sfu"] / per_launch_s / 1e9
    info4 = (ctypes.c_int32 * 4)()
    _lib.check(lib.snp_device_info(info4))
    mhz = clocks.summary().get("sm_mhz") or clocks.summary().get("sm_max_mhz") or 1965.0
    nominal = info4[0] * (64 if args.dtype == "f64" else 128) * 2 * mhz * 1e6 / 1e12   # SMs x FMA lanes x 2 flop x sampled clock
    roofline = {"bound": "fp64" if args.dtype == "f64" else "fp32", "achieved": ach_tflops, "peak": pipe.value, "unit": "TFLOP/s",
                "frac": ach_tflops / pipe.value, "traffic": measured_traffic(args),
                "peak_source": "measured in this run: register-resident FMA loop on all SMs (snp_measure_pipe_peak)",
                "peak_nominal": nominal, "frac_of_nominal": ach_tflops / nominal,
                "peak_nominal_source": f"{info4[0]} SMs x {64 if args.dtype == 'f64' else 128} FMA lanes x 2 x {mhz:.0f} MHz sampled during the timed region",
                "kernel": "snp::k_step (fused 20 sub-steps)", "flops_per_agent_substep": cost["flops"],
                "hbm": {"achieved_gbs": ach_gbs, "peak_gbs": hbm_peak, "frac": ach_gbs / hbm_peak, "peak_source": hbm_src,
                        "bytes_per_agent_step": cost["words"] * wbytes / SUBSTEPS},
                "sfu": {"achieved_gops": ach_sfu, "peak_gops": mufu.value, "frac": ach_sfu / mufu.value if args.dtype == "f32" else None,
                        "ops_per_agent_substep": cost["sfu"]},
                "issue": issue_model(f"{args.workload}:{args.dtype}", clocks.summary(), total_ms / args.steps)}

    line = {"metric": METRIC, "value": value, "unit": "agent-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": workload_config(args.workload, inp),
            "clocks": clocks.summary(), "gpu_launches": launches,
            "e2e": {"value": e2e_value, "unit": "agent-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "CrowdEngine.step_host -> snp_gym_step_host (C ABI, host buffers): pinned H2D action, fused launch whose store phase "
                           "writes observation + flags + reward straight into the pinned host buffers (device-to-host traffic inside the launch), sync",
                    "steps": e2e_steps, "statistic": "median step (host clock around each call), max over ranks",
                    "ms_per_step_median": e2e_med * 1e3, "ms_per_step_mean": e2e_mean * 1e3,
                    "staged_copies_ms_per_step_median": e2e_staged_med * 1e3, "cpu_affinity": affinity_note},
            "roofline": roofline, "wall_s_timed_region": wall, "large_crowd": large}

    if not args.no_cpu_baseline and world == 1:
        if full_affinity:
            os.sched_setaffinity(0, full_affinity)  # the CPU baseline uses every core the job may use
        threads = host_threads()
        n_envs = min(E, max(threads * 4, 128))
        oracle_rate(inp, n_envs, threads, 2)
        reps, spent, done = 0, 0.0, 0
        while spent < (3.0 if ref_baseline else 10.0) and reps < 200:
            _, t = oracle_rate(inp, n_envs, threads, SUBSTEPS)
            spent += t; reps += 1; done += n_envs * N * SUBSTEPS
        port = {"value": done / spent, "unit": "agent-steps/s", "cores": threads, "kind": "port",
                "sample": f"{reps} x ({n_envs} of {E} envs x {SUBSTEPS} sub-steps), oracle/snp_oracle.c (C restatement of the "
                          f"serial Python/NumPy path), OpenMP over envs"}
        # the live reference is the baseline; the C port of the same algorithm is kept beside it as the "compiled CPU" figure
        line["cpu_baseline"] = dict(ref_baseline, c_port=port) if ref_baseline else port
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
