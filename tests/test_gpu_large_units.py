"""The tiled path with partial sums sized for the units in reach (unit_capacity, SNP_OPT_UNIT_SCRATCH), scratch poisoned (0xFF)
before every call:

* LargeCrowd with ample slots, none and half the units listed equals the default-size run bit for bit -- state, goals, robot, flags,
  checks, clock -- for every culled model in fp64 and fp32, on a 4096-human crowd in patch order and the ragged ~1500-human crowd,
  with the example walls, a visible holonomic robot, both checks and 20 sub-steps in one call; the unit counts say what happened;
* TiledCrowdEngine the same at E x N = 5 x 513, 3 x 1000 and 4 x 1024;
* "auto" grows after a call that overflowed, with the same bits throughout;
* 1,500,625 humans in fp64 on one GPU, which the default scratch cannot hold, against default-size runs of three of its slices;
* agent-sharded runs with too few slots on every rank (tests/multi_gpu_units_check.py, two GPUs or more)."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from test_gpu_large_parity import _example_crowd, _f32, _poison
from test_gpu_large_robot import _robot_row

pytestmark = pytest.mark.gpu

DT = 0.0125
ROBOT_SAFETY = 0.05
ACTION = np.array([0.9, 0.35])
CULLED = ["sfm_helbing", "sfm_guo", "hsfm_farina", "hsfm_guo", "hsfm_new", "hsfm_new_guo"]
HERE = os.path.dirname(os.path.abspath(__file__))


@functools.lru_cache(maxsize=None)
def _patch4096():
    """64 x 64 jittered grid over ~128 m (culling leaves a fraction of the units), numbered patch by patch, moving, per-human safety."""
    from social_navigation_pyenvs_b200 import scenarios
    sc = scenarios.jittered_grid_crowd(64, pitch=2.0, jitter=0.5, seed=11)
    S, G = sc["states"][0], sc["goals"][0]
    perm = scenarios.spatial_order(S[:, 0:2])
    S, G = np.ascontiguousarray(S[perm]), np.ascontiguousarray(G[perm])
    rng = np.random.RandomState(12)
    S[:, 5:7] = rng.uniform(-0.6, 0.6, (S.shape[0], 2))
    c, s = np.cos(S[:, 2]), np.sin(S[:, 2])
    S[:, 3], S[:, 4] = c * S[:, 5] - s * S[:, 6], s * S[:, 5] + c * S[:, 6]
    return S, G, rng.uniform(0.0, 0.1, S.shape[0]), scenarios.pack_walls(scenarios.EXAMPLE_WALLS)


def _scene(which, dtype):
    S, G, saf, walls = _patch4096() if which == 4096 else _example_crowd()
    robot = _robot_row(S)
    if dtype == torch.float32:
        S, G, saf, walls, robot = _f32(S, G, saf, walls, robot)
    return S, G, saf, walls, robot


def _large_run(model, scene, dtype, cap, calls=(20,)):
    """A LargeCrowd of the scene stepped `calls` gym steps (visible holonomic robot, both checks); its results after each."""
    from social_navigation_pyenvs_b200.large import LargeCrowd
    S, G, saf, walls, robot = scene
    crowd = LargeCrowd(model, S, G, walls=walls, safety=saf, dtype=dtype, robot=robot, robot_safety=ROBOT_SAFETY, consider_robot=True,
                       unit_capacity=cap)
    out = []
    for k in calls:
        _poison(crowd, True)
        crowd.step(DT, n_substeps=k, action=ACTION, pre_checks=True, post_checks=True)
        e = crowd.eng
        out.append(([t.clone() for t in (e.dyn, e.goal_idx, e.robot, e.flags, e.checks, e.time_now)], crowd.unit_stats()))
    return crowd, out


def _same(a, b, what):
    names = ("dyn", "goal_idx", "robot", "flags", "checks", "time_now")
    for n, x, y in zip(names, a, b):
        assert torch.equal(x, y), f"{what}: {n} differs"


@pytest.mark.parametrize("which", [4096, "ragged"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("model", CULLED)
def test_large_crowd_equals_the_default_run_whatever_the_capacity(model, dtype, which):
    scene = _scene(which, dtype)
    _, [(ref, st0)] = _large_run(model, scene, dtype, None)
    assert st0 == {"capacity": None, "max_listed": None, "fallback_units": None}  # the default size keeps no counts
    n_all = (-(-scene[0].shape[0] // 128)) ** 2
    _, [(got, st)] = _large_run(model, scene, dtype, n_all)  # a slot for every unit
    _same(got, ref, f"{model} {which} capacity {n_all}")
    most = st["max_listed"]
    assert 0 < most <= n_all and st["fallback_units"] == 0, st
    for cap in (most, 0, most // 2):
        _, [(got, st)] = _large_run(model, scene, dtype, cap)
        _same(got, ref, f"{model} {which} capacity {cap}")
        assert st["capacity"] == cap and st["max_listed"] == most, (cap, st)
        if cap == most:
            assert st["fallback_units"] == 0, st
        elif cap == 0:
            assert st["fallback_units"] >= most > 0, st
        else:
            assert st["fallback_units"] >= most - cap > 0, st


def _batch_run(model, N, E, dtype, cap):
    from test_gpu_large_batch import _actions, _batch, _envs
    S, G, saf, walls, robots = _envs(N)
    S, G, saf, robots = S[:E], G[:E], saf[:E], robots[:E]
    act = _actions("holonomic")[:E]
    if dtype == torch.float32:
        S, G, saf, walls, robots, act = _f32(S, G, saf, walls, robots, act)
    from social_navigation_pyenvs_b200 import TiledCrowdEngine
    eng = TiledCrowdEngine.from_reference_arrays(model, S, G, walls=walls, safety=saf, robot=robots, dtype=dtype, unit_capacity=cap)
    eng.set_robot_rows(robots, safety=np.full(len(robots), ROBOT_SAFETY))
    eng.consider_robot = True
    out = []
    for k in (3, 2):
        eng.scratch.fill_(0xFF)
        eng.step(act, DT, n_substeps=k, pre_checks=True, post_checks=True)
        out.append(([t.clone() for t in (eng.dyn, eng.goal_idx, eng.robot, eng.flags, eng.checks, eng.time_now)], eng.unit_stats()))
    return out


@pytest.mark.parametrize("E,N", [(5, 513), (3, 1000), (4, 1024)])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("model", ["sfm_helbing", "hsfm_new_guo"])
def test_tiled_engine_equals_the_default_run_whatever_the_capacity(model, dtype, E, N):
    ref = _batch_run(model, N, E, dtype, None)
    full = _batch_run(model, N, E, dtype, E * (-(-N // 128)) ** 2)  # a slot for every unit
    for (g, st), (r, _) in zip(full, ref):
        _same(g, r, f"{model} {E}x{N} every unit with a slot")
        assert st["fallback_units"] == 0, st
    most = max(st["max_listed"] for _, st in full)
    for cap in (most, 0, most // 2):
        got = _batch_run(model, N, E, dtype, cap)
        for (g, st), (r, _) in zip(got, ref):
            _same(g, r, f"{model} {E}x{N} capacity {cap}")
        if cap == 0:
            assert all(st["fallback_units"] >= st["max_listed"] > 0 for _, st in got)
        elif cap == most:
            assert all(st["fallback_units"] == 0 for _, st in got)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
def test_auto_capacity_grows_after_an_overflow(dtype, monkeypatch):
    """Two slots per agent block to start with: the first call overflows and the finish kernel evaluates the rest; the second has
    ceil(1.25 x the most listed) slots and none left over.  The same bits as the default run after each call."""
    from social_navigation_pyenvs_b200 import large
    monkeypatch.setattr(large, "AUTO_UNITS_PER_BLOCK", 2)
    scene = _scene(4096, dtype)
    _, ref = _large_run("hsfm_farina", scene, dtype, None, calls=(20, 5))
    crowd, got = _large_run("hsfm_farina", scene, dtype, "auto", calls=(20, 5))
    (g1, st1), (g2, st2) = got
    _same(g1, ref[0][0], "auto, first call")
    _same(g2, ref[1][0], "auto, second call")
    assert st1["capacity"] == 2 * 32 and st1["fallback_units"] > 0, st1
    assert st2["capacity"] == -(-5 * st1["max_listed"] // 4) and st2["fallback_units"] == 0, (st1, st2)


def test_a_crowd_the_default_scratch_cannot_hold():
    """1,500,625 humans (a 1225 x 1225 jittered grid in patch order), fp64, hsfm_farina: the default scratch is larger than the GPU;
    with unit_capacity="auto" one sub-step runs in a scratch below 4 GB, and three tile-aligned 4096-human slices (first, middle,
    last) equal default-size runs of those slices (shard=) bit for bit."""
    from social_navigation_pyenvs_b200 import _lib as L, scenarios
    from social_navigation_pyenvs_b200.large import LargeCrowd
    n_side = 1225
    n = n_side * n_side
    assert int(L.lib().snp_large_scratch_bytes(n, n, L.SNP_F64)) > torch.cuda.get_device_properties(0).total_memory
    sc = scenarios.jittered_grid_crowd(n_side, pitch=2.0, jitter=0.5, seed=21)
    S, G = sc["states"][0], sc["goals"][0]
    perm = scenarios.spatial_order(S[:, 0:2])
    S, G = np.ascontiguousarray(S[perm]), np.ascontiguousarray(G[perm])
    S[:, 3:5] = S[:, 5:7] = np.random.RandomState(22).uniform(-0.5, 0.5, (n, 2))
    S[:, 2] = 0.0  # heading 0: the body and world velocities agree
    big = LargeCrowd("hsfm_farina", S, G, dtype=torch.float64, unit_capacity="auto")
    big.scratch.fill_(0xFF)
    cap = big.unit_capacity
    assert big.scratch.numel() < 4 * 2 ** 30
    big.step(DT, n_substeps=1)
    st = big.unit_stats()
    print(f"1,500,625 humans fp64: capacity {st['capacity']}, listed {st['max_listed']}, evaluated by the finish kernel "
          f"{st['fallback_units']}, scratch {big.scratch.numel() / 2 ** 30:.2f} GiB")
    assert st["capacity"] == cap and st["max_listed"] > 0
    dyn, gidx = big.eng.dyn[:, 0], big.eng.goal_idx[0]
    for off in (0, (n // 2) // 128 * 128, (n - 4096) // 128 * 128):
        part = LargeCrowd("hsfm_farina", S, G, dtype=torch.float64, shard=(off, 4096))
        part.scratch.fill_(0xFF)
        part.step(DT, n_substeps=1)
        assert torch.equal(part.eng.dyn[:, 0], dyn[:, off:off + 4096]), off
        assert torch.equal(part.eng.goal_idx[0], gidx[off:off + 4096]), off
        del part
        torch.cuda.empty_cache()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs of one node")
@pytest.mark.parametrize("ranks", [2, 8])
def test_sharded_with_too_few_slots_equals_single_gpu_bit_for_bit(ranks):
    if torch.cuda.device_count() < ranks:
        pytest.skip(f"{ranks} GPUs needed")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={ranks}", "--master-addr", "127.0.0.1",
           "--master-port", "29557", os.path.join(HERE, "multi_gpu_units_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and f"MULTI_GPU_UNITS_CHECK OK on {ranks} ranks" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
