"""E environments of more than 512 humans each through snp_large_batch_step (TiledCrowdEngine), with the scratch filled with NaN
before every call:

* env e of a batch is bit for bit LargeCrowd(env e) -- rows, robot, flags, checks, clock -- for every model and dtype, N = 513, 1000
  (ragged last tile) and 1024 (whole tiles, boxes folded into the finish kernel), with the envs on top of each other in the plane so
  that a pair across envs would be in reach;
* the oracle on the same E-env batch after one sub-step, and its checks bit for bit;
* culling off == culling on bit for bit, with an env whose every tile is culled;
* per-env walls against the oracle;
* continuity at N = 300 and 512 with the small-crowd engine;
* the laser of a 1000-human batch against the oracle."""
import functools

import numpy as np
import pytest
import torch

import oracle
from oracle import OracleConfig
from test_gpu_large_parity import _crowd_with_walls, _err, _f32, _poison
from test_gpu_large_robot import _robot_row

pytestmark = pytest.mark.gpu

SFMS = oracle.SFMS
DT = 0.0125
E = 5
ROBOT_SAFETY = 0.05


@functools.lru_cache(maxsize=None)
def _envs(N):
    """E seeded, jittered, moving crowds of N humans around the same centre (per-human safety, goal switches), the example walls,
    and one robot per env near its crowd's centre."""
    from social_navigation_pyenvs_b200 import scenarios
    S, G, saf = [], [], []
    for e in range(E):
        s, g, sf = _crowd_with_walls(scenarios.EXAMPLE_WALLS, 0.7, seed=7 + e)
        S.append(s[:N]); G.append(g[:N]); saf.append(sf[:N])
    S, G, saf = np.stack(S), np.stack(G), np.stack(saf)
    robots = np.stack([_robot_row(S[e], yaw=0.4 + 0.5 * e) for e in range(E)])
    return S, G, saf, scenarios.pack_walls(scenarios.EXAMPLE_WALLS), robots


def _actions(kinematics):
    if kinematics == "holonomic":
        return np.array([[0.9 - 0.1 * e, 0.35 - 0.2 * e] for e in range(E)])
    return np.array([[0.8 - 0.05 * e, 0.05 - 0.02 * e] for e in range(E)])


def _batch(model, S, G, saf, walls, robots, dtype, consider_robot=True):
    from social_navigation_pyenvs_b200 import TiledCrowdEngine
    eng = TiledCrowdEngine.from_reference_arrays(model, S, G, walls=walls, safety=saf, robot=robots, dtype=dtype)
    eng.set_robot_rows(robots, safety=np.full(len(robots), ROBOT_SAFETY))
    eng.consider_robot = consider_robot  # the robot is not a row of the states: only the step options carry it
    return eng


def _batch_step(eng, *args, **kw):
    eng.scratch.fill_(0xFF)  # NaN in both dtypes
    eng.step(*args, **kw)


@pytest.mark.parametrize("N", [513, 1000, 1024])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("model,kinematics,visible", [(m, "holonomic", True) for m in SFMS] +
                         [(m, "unicycle", False) for m in ("sfm_helbing", "hsfm_new_guo", "hsfm_moussaid")])
def test_every_env_equals_its_own_large_crowd_bit_for_bit(model, kinematics, visible, dtype, N):
    """Two gym steps (3 then 2 sub-steps, both checks) of the batch against E LargeCrowds stepped with the same robot and action.
    Every batch call publishes the entity view from the state (v = R(yaw) bv on the device for headed models, where the finish kernel's
    own velocity can differ in the last bit), so each LargeCrowd republishes its view before its step too."""
    from social_navigation_pyenvs_b200.large import LargeCrowd
    S, G, saf, walls, robots = _envs(N)
    act = _actions(kinematics)
    if dtype == torch.float32:
        S, G, saf, walls, robots, act = _f32(S, G, saf, walls, robots, act)
    batch = _batch(model, S, G, saf, walls, robots, dtype, visible)
    singles = [LargeCrowd(model, S[e], G[e], walls=walls, safety=saf[e], dtype=dtype, symmetric=True, robot=robots[e], robot_safety=ROBOT_SAFETY,
                          consider_robot=visible) for e in range(E)]
    for k in (3, 2):
        _batch_step(batch, act, DT, n_substeps=k, pre_checks=True, post_checks=True, kinematics=kinematics)
        for e, one in enumerate(singles):
            _poison(one, True)
            one._publish()  # a batch call publishes the view from the state, as a LargeCrowd built from it does
            one.step(DT, n_substeps=k, action=act[e], kinematics=kinematics, pre_checks=True, post_checks=True)
    rows, (rob, _) = batch.rows(S), batch.robot_rows()
    flags, checks, clock = batch.flags.cpu().numpy(), batch.checks.cpu().numpy(), batch.time_now.cpu().numpy()
    for e, one in enumerate(singles):
        assert np.array_equal(rows[e], one.local_rows(S[e])), e
        assert np.array_equal(rob[e], one.robot_rows()), e
        assert flags[e] == int(one.eng.flags[0]) and np.array_equal(checks[e], one.eng.checks[0].cpu().numpy()), e
        assert clock[e] == float(one.eng.time_now[0]), e
    assert not np.array_equal(rows[0], rows[1])  # the envs are different crowds


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("model", SFMS)
def test_batch_against_the_oracle(model, dtype):
    """One sub-step of the 5 x 1000 batch with a visible holonomic robot against oracle.update_humans on the same batch (the robot as
    row N, robot_vel = action); the pre-step checks (non-headed models: the stored velocity is the view's) and the post-step checks
    on the batch's own end state against oracle.checks bit for bit."""
    S, G, saf, walls, robots = _envs(1000)
    act = _actions("holonomic")
    if dtype == torch.float32:
        S, G, saf, walls, robots, act = _f32(S, G, saf, walls, robots, act)
    n = S.shape[1]
    eng = _batch(model, S, G, saf, walls, robots, dtype)
    consts = np.array(eng.consts)
    _batch_step(eng, act, DT, n_substeps=1, pre_checks=True, post_checks=True)
    f = eng.decode_flags()
    cfg = OracleConfig(oracle.type_code(model), True, True, False)
    Sr = np.concatenate([S, robots[:, None]], 1)
    saf_r = np.concatenate([saf, np.full((E, 1), ROBOT_SAFETY)], 1)
    ref, _, _ = oracle.update_humans(cfg, Sr, G, walls, np.tile(oracle.default_params(model), (E, n, 1)), saf_r, np.zeros((E, n, 2)), DT, 1,
                                     robot_vel=act, n_threads=8)
    got = eng.rows(S)
    err = max(_err(got[e], ref[e, :n]) for e in range(E))
    assert err <= (1e-9 if dtype == torch.float64 else 1e-4), err
    for e in range(E):
        assert np.array_equal(got[e][:, 10:12], ref[e, :n, 10:12])
    rob = eng.robot_rows()[0]
    post = oracle.checks(got, n, rob, act, eng.time_now.cpu().numpy(), consts)
    assert np.array_equal(f["actual_collision"], post[:, 7] != 0) and np.array_equal(f["actual_dmin"], post[:, 8])
    assert np.array_equal(f["actual_goal"], post[:, 9] != 0)
    if not model.startswith("hsfm"):
        pre = oracle.checks(S, n, robots, act, np.zeros(E), consts)
        assert np.array_equal(f["collision"], pre[:, 0] != 0) and np.array_equal(f["dmin"], pre[:, 1])
        assert np.array_equal(f["reaching_goal"], pre[:, 2] != 0) and np.array_equal(f["reward"], pre[:, 3])
        assert np.array_equal(f["info"], pre[:, 6].astype(int))


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("model", ["sfm_helbing", "hsfm_farina"])
def test_culling_off_equals_culling_on_with_an_env_that_culls_everything(model, dtype):
    """Env 0's humans stand 80 m apart (beyond the culling reach, every tile is culled); the others are dense.  Culling on and off
    give the same bits, in three sub-steps and the robot's checks."""
    S, G, saf, walls, robots = _envs(1000)
    S, G, saf, robots = S.copy(), G.copy(), saf.copy(), robots.copy()
    n = S.shape[1]
    ix, iy = np.meshgrid(np.arange(32), np.arange(32), indexing="ij")
    S[0, :, 0], S[0, :, 1] = 80.0 * ix.ravel()[:n] + 500.0, 80.0 * iy.ravel()[:n]
    G[0] = S[0, :, None, 0:2] + [3.0, 1.0]
    S[0, :, 10:12] = G[0, :, 0]
    act = _actions("holonomic")
    if dtype == torch.float32:
        S, G, saf, walls, robots, act = _f32(S, G, saf, walls, robots, act)
    out = []
    for culling in (True, False):
        eng = _batch(model, S, G, saf, walls, robots, dtype)
        eng.culling = culling
        _batch_step(eng, act, DT, n_substeps=3, pre_checks=True, post_checks=True)
        out.append((eng.rows(S), eng.robot_rows()[0], eng.flags.cpu().numpy(), eng.checks.cpu().numpy()))
    for a, b in zip(*out):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("model", ["sfm_guo", "hsfm_farina", "hsfm_new_moussaid"])
def test_per_env_walls_against_the_oracle(model, dtype):
    """walls [E,W,S,2,2]: env e gets the example walls shifted by e * 0.1 m (so that every env's humans meet other walls); one
    sub-step against the oracle with the same per-env walls, and the batch differs from the one with shared walls."""
    S, G, saf, walls, robots = _envs(1000)
    wall_e = np.stack([walls + 0.1 * e for e in range(E)])
    act = _actions("holonomic")
    if dtype == torch.float32:
        S, G, saf, wall_e, robots, act = _f32(S, G, saf, wall_e, robots, act)
    n = S.shape[1]
    eng = _batch(model, S, G, saf, wall_e, robots, dtype, consider_robot=False)
    _batch_step(eng, act, DT, n_substeps=1, pre_checks=False)
    cfg = OracleConfig(oracle.type_code(model), False, True, False)
    ref, _, _ = oracle.update_humans(cfg, S, G, wall_e, np.tile(oracle.default_params(model), (E, n, 1)), saf, np.zeros((E, n, 2)), DT, 1, n_threads=8)
    got = eng.rows(S)
    err = max(_err(got[e], ref[e]) for e in range(E))
    assert err <= (1e-9 if dtype == torch.float64 else 1e-4), err
    shared = _batch(model, S, G, saf, wall_e[0], robots, dtype, consider_robot=False)
    _batch_step(shared, act, DT, n_substeps=1, pre_checks=False)
    assert np.array_equal(shared.rows(S)[0], got[0]) and not np.array_equal(shared.rows(S)[1], got[1])


@pytest.mark.parametrize("N", [300, 512])
@pytest.mark.parametrize("model", ["sfm_helbing", "hsfm_farina", "hsfm_new_moussaid"])
def test_continuity_with_the_small_crowd_engine(model, N):
    """Where both engines apply, TiledCrowdEngine and CrowdEngine load the same arrays (the robot as a visible row) and step alike:
    two gym steps of 2 sub-steps with both checks; the humans within 1e-12 relative (the summation orders differ), the robot and
    the clock bit for bit, the first step's flags identical."""
    from social_navigation_pyenvs_b200 import CrowdEngine, TiledCrowdEngine
    S, G, saf, walls, robots = _envs(N)
    act = _actions("holonomic")
    Sr = np.concatenate([S, robots[:, None]], 1)
    saf_r = np.concatenate([saf, np.full((E, 1), ROBOT_SAFETY)], 1)
    engines = [cls.from_reference_arrays(model, Sr, G, walls=walls, safety=saf_r, consider_robot=True) for cls in (CrowdEngine, TiledCrowdEngine)]
    for step in range(2):
        flags = []
        for eng in engines:
            if isinstance(eng, TiledCrowdEngine):
                eng.scratch.fill_(0xFF)
            eng.step(act, DT, n_substeps=2, pre_checks=True, post_checks=True)
            flags.append(eng.flags.cpu().numpy())
        if step == 0:
            assert np.array_equal(flags[0], flags[1])
        small, tiled = engines
        assert np.array_equal(small.robot_rows()[0], tiled.robot_rows()[0])
        assert np.array_equal(small.time_now.cpu().numpy(), tiled.time_now.cpu().numpy())
    a, b = engines[0].rows(Sr)[:, :N], engines[1].rows(Sr)[:, :N]
    err = max(_err(b[e], a[e]) for e in range(E))
    assert err < 1e-12, err


def test_laser_scan_of_a_1000_human_batch_against_the_oracle():
    """sensors.EngineScanner over a TiledCrowdEngine of 5 x 1000 humans (snp_laser switches to one warp per ray above 512 entities)
    after a step: ranges within 1e-11 of oracle.laser's, hit indices exact."""
    from social_navigation_pyenvs_b200.sensors import EngineScanner
    S, G, saf, walls, robots = _envs(1000)
    eng = _batch("hsfm_farina", S, G, saf, walls, robots, torch.float64)
    _batch_step(eng, _actions("holonomic"), DT, n_substeps=3, pre_checks=True)
    rob = eng.robot_rows()[0]
    pose = torch.as_tensor(np.ascontiguousarray(rob[:, [0, 1, 2]].T), dtype=torch.float64, device=eng.device)
    ranges, hits = EngineScanner(eng, 2 * np.pi, 360, 10.0).scan(pose)
    rows = eng.rows(S)
    ref_r, ref_h = oracle.laser(rows[:, :, [0, 1, 8]], walls, rob[:, [0, 1, 2]], 2 * np.pi, 360, 10.0)
    assert np.abs(ranges.cpu().numpy() - ref_r).max() < 1e-11
    assert np.array_equal(hits.cpu().numpy().astype(np.int64), ref_h)
    assert (hits.cpu().numpy() >= 0).sum() > 100 * E
