"""The robot of SocialNavGym.step in the large crowd (LargeCrowd(robot=...)): its force on the humans and its motion inside
snp_large_run_p2p, the checks of snp_large_checks and the laser -- with the scratch and the tile boxes poisoned before every step
call, as in test_gpu_large_parity.py:

* a visible robot crossing the moving ~1500-human crowd (ragged last tile, example walls, per-human safety) against the oracle,
  every model in fp64 and fp32, holonomic and unicycle;
* an invisible robot leaves the humans bit for bit as without it;
* the checks bit for bit against the oracle's, every info code, with the first colliding human in a later tile than a nearer one;
* a second witness: the small-crowd engine with the same robot and action;
* shard= slices and one sub-step per call: the same bits; the laser against the oracle's."""
import functools

import numpy as np
import pytest
import torch

import oracle
from oracle import OracleConfig
from helpers import rel_err, unicycle_step, wrap_angle_cols
from test_gpu_large_parity import _check, _err, _example_crowd, _f32, _grid72, _poison

pytestmark = pytest.mark.gpu

SFMS = oracle.SFMS
DT = 0.0125
ROBOT_SAFETY = 0.05
CONSTS = np.array([50.0, -0.25, 1.0, 0.2, 0.5, 0.25])


def _step(crowd, k, whole=True, **kw):
    _poison(crowd, whole)
    crowd.step(DT, n_substeps=k, **kw)


def _robot_row(S, yaw=0.4):
    """A robot of radius 0.3 near the crowd's centre whose nearest human is 0.8 m away (well within every pair law's reach, not
    overlapping), its goal 4 m ahead."""
    c = np.linspace(-3.0, 3.0, 61)
    cand = np.stack(np.meshgrid(c, c, indexing="ij"), -1).reshape(-1, 2) + S[:, 0:2].mean(0)
    gap = np.min(np.hypot(cand[:, None, 0] - S[None, :, 0], cand[:, None, 1] - S[None, :, 1]), 1)
    p = cand[np.argmin(np.abs(gap - 0.8))]
    r = np.zeros(13)
    r[0:2], r[2], r[8], r[9], r[12] = p, yaw, 0.3, 80.0, 1.0
    r[10:12] = p + [4.0, 0.0]
    return r


def _large(model, S, G, dtype, robot, consider_robot=True, **kw):
    from social_navigation_pyenvs_b200.large import LargeCrowd
    return LargeCrowd(model, S, G, dtype=dtype, symmetric=True, robot=robot, robot_safety=ROBOT_SAFETY, consider_robot=consider_robot, **kw)


def _oracle_holonomic(model, S, G, walls, safety, action, k, D=None):
    """k sub-steps of the oracle with the robot as row n (holonomic action before every sub-step)."""
    n = S.shape[0] - 1
    cfg = OracleConfig(oracle.type_code(model), True, True, False)
    params = np.tile(oracle.default_params(model), (1, n, 1))
    saf = np.concatenate([safety, [ROBOT_SAFETY]])[None]
    D = np.zeros((1, n, 2)) if D is None else D
    ref, Gr, Dr = oracle.update_humans(cfg, S[None], G[None], walls, params, saf, D, DT, k, robot_vel=np.asarray(action)[None], n_threads=8)
    return ref[0], Gr[0], Dr


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("model", SFMS)
def test_visible_holonomic_robot_against_the_oracle(model, dtype):
    """The robot's pair force (entity M, after the chunk sums; Moussaid with the human as agent 1) and its holonomic motion
    recomputed by every finish thread: 3 sub-steps, then 2 more in a second call (fp32 also one sub-step), against the oracle with
    robot_vel; the robot's end state too."""
    S, G, safety, walls = _example_crowd()
    robot = _robot_row(S)
    action = np.array([0.9, 0.35])
    if dtype == torch.float32:
        S, G, walls, safety, robot, action = _f32(S, G, walls, safety, robot, action)
    Sr = np.concatenate([S, robot[None]])
    ref3, G3, D3 = _oracle_holonomic(model, Sr, G, walls, safety, action, 3)
    ref5, _, _ = _oracle_holonomic(model, ref3, G3, walls, safety, action, 2, D3)
    n = S.shape[0]
    errs = {}
    if dtype == torch.float32:
        ref1, _, _ = _oracle_holonomic(model, Sr, G, walls, safety, action, 1)
        one = _large(model, S, G, dtype, robot, walls=walls, safety=safety)
        _step(one, 1, action=action)
        errs["1"] = _err(one.local_rows(S), ref1[:n])
    crowd = _large(model, S, G, dtype, robot, walls=walls, safety=safety)
    _step(crowd, 3, action=action)
    got3 = crowd.local_rows(S)
    _step(crowd, 2, action=action)
    got5 = crowd.local_rows(S)
    errs["3"], errs["5"] = _err(got3, ref3[:n]), _err(got5, ref5[:n])
    assert np.array_equal(got5[:, 10:12], ref5[:n, 10:12])
    # the robot moved through the crowd and pushed somebody: without it the humans end elsewhere
    bare = _large(model, S, G, dtype, robot, consider_robot=False, walls=walls, safety=safety)
    _step(bare, 5, action=action)
    assert not np.array_equal(bare.local_rows(S), got5)
    rb = crowd.robot_rows()
    tol = 1e-12 if dtype == torch.float64 else 1e-5
    assert np.abs(rb[0:2] - ref5[n, 0:2]).max() < tol and np.array_equal(rb[3:5], ref5[n, 3:5])
    print(f"large robot parity {model} {str(dtype)[6:]}: " + " ".join(f"{k} sub-steps {v:.2e}" for k, v in errs.items()))
    _check(model, dtype, errs)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("model", ["sfm_helbing", "hsfm_new_guo", "hsfm_moussaid"])
def test_visible_unicycle_robot_against_the_oracle(model, dtype):
    """robot_mode 3: the oracle stepped one sub-step at a time around helpers.unicycle_step (the robot row moved in NumPy)."""
    S, G, safety, walls = _example_crowd()
    robot = _robot_row(S, yaw=2.9)
    action = np.array([0.8, 0.05])  # (v, r): r is added at every sub-step
    if dtype == torch.float32:
        S, G, walls, safety, robot, action = _f32(S, G, walls, safety, robot, action)
    n, k = S.shape[0], 5
    cfg = OracleConfig(oracle.type_code(model), True, True, False)
    params = np.tile(oracle.default_params(model), (1, n, 1))
    saf = np.concatenate([safety, [ROBOT_SAFETY]])[None]
    Sr, Gr, D = np.concatenate([S, robot[None]])[None], G[None], np.zeros((1, n, 2))
    yaw = robot[2]
    for _ in range(k):
        Sr[0, n, 0:2], yaw, Sr[0, n, 3:5] = unicycle_step(Sr[0, n, 0:2], yaw, action[0], action[1], DT)
        Sr, Gr, D = oracle.update_humans(cfg, Sr, Gr, walls, params, saf, D, DT, 1, n_threads=8)
    crowd = _large(model, S, G, dtype, robot, walls=walls, safety=safety)
    _step(crowd, k, action=action, kinematics="unicycle")
    e = _err(crowd.local_rows(S), Sr[0, :n])
    tol = (1e-6 if "moussaid" in model else 1e-9) if dtype == torch.float64 else (5e-3 if model.startswith("hsfm_new") else 5e-4)
    assert e < tol, (model, e)
    rb = crowd.robot_rows()
    rtol = 1e-12 if dtype == torch.float64 else 1e-5
    assert np.abs(rb[0:2] - Sr[0, n, 0:2]).max() < rtol and abs(rb[2] - yaw) < rtol and np.abs(rb[3:5] - Sr[0, n, 3:5]).max() < rtol


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("kinematics", ["holonomic", "unicycle"])
def test_invisible_robot_leaves_the_humans_bit_for_bit(kinematics, dtype):
    """consider_robot=False: the robot moves (and the clock runs) but the humans are exactly those of the crowd without a robot."""
    from social_navigation_pyenvs_b200.large import LargeCrowd
    S, G, safety, walls = _example_crowd()
    robot = _robot_row(S)
    plain = LargeCrowd("hsfm_farina", S, G, walls=walls, safety=safety, dtype=dtype)
    _step(plain, 4)
    ghost = _large("hsfm_farina", S, G, dtype, robot, consider_robot=False, walls=walls, safety=safety)
    _step(ghost, 4, action=[0.9, 0.2], kinematics=kinematics, pre_checks=True, post_checks=True)
    assert np.array_equal(ghost.local_rows(S), plain.local_rows(S))
    assert not np.array_equal(ghost.robot_rows()[0:2], robot[0:2])
    assert float(ghost.eng.time_now[0]) == DT + DT + DT + DT


# ---- the checks: bit for bit ----

def _checks_crowd(case, M):
    """M resting humans (sfm: the view's velocity is the stored one) far from a robot at the origin, then per case: humans placed in
    its path.  Returns (states, goals, robot, action, time_now)."""
    rng = np.random.RandomState(11)
    S = np.zeros((M, 13))
    ang = rng.uniform(0, 2 * np.pi, M)
    rad = rng.uniform(3.0, 30.0, M)
    S[:, 0], S[:, 1] = rad * np.cos(ang), rad * np.sin(ang)
    S[:, 3:5] = rng.uniform(-0.5, 0.5, (M, 2))
    S[:, 8], S[:, 9], S[:, 12] = rng.uniform(0.25, 0.35, M), 75.0, 1.0
    S[:, 10:12] = S[:, 0:2]
    robot = np.zeros(13)
    robot[8], robot[9], robot[12] = 0.3, 80.0, 1.0
    robot[10:12] = [20.0, 20.0]
    action, t = np.array([1.0, 0.0]), 0.0
    if case == "timeout":
        t = 49.25
    elif case == "collision_late_tile":
        # human 900 (tile 7) is swept into; humans 5 (tile 0) and 700 (tile 5) come near but do not touch (dmin); human 910,
        # after the colliding one, nearer still -- the sweep has stopped before it
        S[5, 0:2], S[5, 3:5], S[5, 8] = [0.1, 0.95], [0.0, 0.0], 0.3
        S[700, 0:2], S[700, 3:5], S[700, 8] = [0.2, -0.9], [0.0, 0.0], 0.3
        S[900, 0:2], S[900, 3:5], S[900, 8] = [0.5, 0.6], [0.0, -0.5], 0.3
        S[910, 0:2], S[910, 3:5], S[910, 8] = [-0.2, 0.62], [0.0, 0.0], 0.3
    elif case == "goal":
        robot[10:12] = [0.25, 0.0]
    elif case == "danger":
        S[300, 0:2], S[300, 3:5], S[300, 8] = [0.0, 0.7], [0.0, 0.0], 0.3
    return S, np.repeat(S[:, None, 0:2], 2, 1), robot, action, t


@pytest.mark.parametrize("M", [1000, 1030, 4096])
@pytest.mark.parametrize("case", ["nothing", "timeout", "collision_late_tile", "goal", "danger"])
def test_checks_bit_for_bit_against_the_oracle(case, M):
    """Flags, dmin, reward, info code and the actual checks == oracle.checks bit for bit (info codes 0..4).  M = 1030 is not a
    multiple of 128; 4096 gives every thread of the checks CTA four humans."""
    S, G, robot, action, t = _checks_crowd(case, M)
    crowd = _large("sfm_helbing", S, G, torch.float64, robot)
    crowd.eng.time_now.fill_(t)
    crowd.eng.consts = list(CONSTS)
    crowd.step(DT, n_substeps=0, action=action, pre_checks=True, post_checks=True)
    f = crowd.decode_flags()
    ref = oracle.checks(S[None], M, robot[None], action[None], np.array([t]), CONSTS)[0]
    assert int(f["info"][0]) == {"nothing": 0, "timeout": 1, "collision_late_tile": 2, "goal": 3, "danger": 4}[case]
    assert bool(f["collision"][0]) == bool(ref[0]) and bool(f["reaching_goal"][0]) == bool(ref[2])
    assert f["dmin"][0] == ref[1] and f["reward"][0] == ref[3]
    assert (bool(f["terminated"][0]), bool(f["truncated"][0]), int(f["info"][0])) == (bool(ref[4]), bool(ref[5]), int(ref[6]))
    assert bool(f["actual_collision"][0]) == bool(ref[7]) and f["actual_dmin"][0] == ref[8] and bool(f["actual_goal"][0]) == bool(ref[9])
    if case == "collision_late_tile":
        d5 = np.hypot(0.1, 0.95) - 0.6
        assert 0.2 < f["dmin"][0] <= d5  # human 910, after the colliding one, would give 0.05


# ---- a second witness: the small-crowd engine ----

@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("model", ["sfm_helbing", "hsfm_farina"])
def test_same_robot_and_checks_as_the_small_crowd_engine(model, dtype):
    """500 humans through LargeCrowd and through CrowdEngine(E=1, N=500), a visible holonomic robot, two gym steps of 20 sub-steps
    with both checks.  The robot's end state, the clock and every flag are bit-identical (the same expressions), the humans within
    tolerance (different summation order).  The first step's swept check is bit-identical for sfm; a headed model's view velocity is
    R(yaw) bv computed on the device, which can differ in the last bit from the host-loaded velocity the small engine checks with."""
    from social_navigation_pyenvs_b200 import CrowdEngine
    sc = _grid72("row")
    S, G = np.ascontiguousarray(sc[0][:500]), np.ascontiguousarray(sc[1][:500])
    c, s = np.cos(S[:, 2]), np.sin(S[:, 2])
    S[:, 3], S[:, 4] = c * S[:, 5] - s * S[:, 6], s * S[:, 5] + c * S[:, 6]  # v = R(yaw) bv, as the engines keep it
    robot = _robot_row(S)
    action = np.array([0.6, 0.25])
    if dtype == torch.float32:
        S, G, robot, action = _f32(S, G, robot, action)
    saf = np.concatenate([np.zeros(500), [ROBOT_SAFETY]])[None]
    small = CrowdEngine.from_reference_arrays(model, np.concatenate([S, robot[None]])[None], G[None], consider_robot=True, safety=saf, dtype=dtype)
    large = _large(model, S, G, dtype, robot)
    for step in range(2):
        small.step(action[None], DT, n_substeps=20, pre_checks=True, post_checks=True)
        _step(large, 20, action=action, pre_checks=True, post_checks=True)
        fs, fl = small.decode_flags(), large.decode_flags()
        for key in ("collision", "reaching_goal", "terminated", "truncated", "info", "actual_collision", "actual_goal"):
            assert np.array_equal(fs[key], fl[key]), (step, key)
        if step == 0 and model == "sfm_helbing":
            assert fs["dmin"][0] == fl["dmin"][0] and fs["reward"][0] == fl["reward"][0]
        else:
            assert abs(fs["dmin"][0] - fl["dmin"][0]) <= (1e-9 if dtype == torch.float64 else 1e-4)
        assert np.array_equal(small.robot_rows()[0][0], large.robot_rows())
        assert float(small.time_now[0]) == float(large.eng.time_now[0])
    got, ref = large.local_rows(S), small.rows(np.concatenate([S, robot[None]])[None])[0, :500]
    err = float(rel_err(wrap_angle_cols(got[:, :8], ref[:, :8]), ref[:, :8]).max())
    assert err < (1e-9 if dtype == torch.float64 else 5e-3), err


# ---- slices, calls and exchanges: bit for bit ----

@functools.lru_cache(maxsize=None)
def _whole_robot_after_one(dtype):
    S, G = _grid72("patch")
    crowd = _large("hsfm_farina", S, G, dtype, _robot_row(S))
    _step(crowd, 1, action=[0.7, -0.3])
    return crowd.local_rows(S)


@pytest.mark.parametrize("shard", [(0, 1000), (64, 72 * 72 - 64), (1024, 1024)], ids=["0+1000", "64+rest", "1024+1024"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
def test_robot_slices_same_bits_as_the_whole_crowd(dtype, shard):
    """A shard= slice with the robot (every rank recomputes it): after one sub-step its rows are the whole crowd's."""
    S, G = _grid72("patch")
    off, n = shard
    crowd = _large("hsfm_farina", S, G, dtype, _robot_row(S), shard=shard)
    _step(crowd, 1, whole=False, action=[0.7, -0.3])
    assert np.array_equal(crowd.local_rows(S[off:off + n]), _whole_robot_after_one(dtype)[off:off + n])


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("kinematics", ["holonomic", "unicycle"])
def test_robot_sub_steps_in_one_call_equal_one_per_call_and_nccl(kinematics, dtype):
    """k sub-steps in one call == k calls of one == the NCCL exchange forced on one GPU (one call per sub-step, the robot and the
    clock carried between calls): humans, robot and time_now bit for bit."""
    S, G = _grid72("patch")
    robot = _robot_row(S)
    act = [0.7, -0.3] if kinematics == "holonomic" else [0.7, 0.04]
    one = _large("hsfm_farina", S, G, dtype, robot)
    _step(one, 5, action=act, kinematics=kinematics)
    many = _large("hsfm_farina", S, G, dtype, robot)
    for _ in range(5):
        _step(many, 1, action=act, kinematics=kinematics)
    nccl = _large("hsfm_farina", S, G, dtype, robot, exchange="nccl")
    assert nccl.exchange == "nccl"
    _step(nccl, 5, action=act, kinematics=kinematics)
    for other in (many, nccl):
        assert np.array_equal(one.local_rows(S), other.local_rows(S))
        assert np.array_equal(one.robot_rows(), other.robot_rows())
        assert float(one.eng.time_now[0]) == float(other.eng.time_now[0])


# ---- the laser ----

def test_laser_scan_against_the_oracle():
    """LargeCrowd.scan = snp_laser over the view's positions, the static radii and the walls from the robot's pose: ranges within
    1e-11 of the oracle's, hit indices (global human index, M + segment ordinal) exact."""
    S, G, safety, walls = _example_crowd()
    robot = _robot_row(S, yaw=0.3)
    crowd = _large("hsfm_farina", S, G, torch.float64, robot, walls=walls, safety=safety)
    _step(crowd, 3, action=[0.5, 0.1])
    ranges, hits = crowd.scan(2 * np.pi, 360, 10.0)
    v = crowd.view[crowd.cur].double().cpu().numpy()
    humans = np.stack([v[0], v[1], S[:, 8]], 1)[None]
    rb = crowd.robot_rows()
    ref_r, ref_h = oracle.laser(humans, walls, rb[None, [0, 1, 2]], 2 * np.pi, 360, 10.0)
    assert np.abs(ranges.cpu().numpy() - ref_r[0]).max() < 1e-11
    assert np.array_equal(hits.cpu().numpy().astype(np.int64), ref_h[0])
    assert (hits.cpu().numpy() >= 0).sum() > 100
