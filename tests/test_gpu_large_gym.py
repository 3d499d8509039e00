"""The batched gym beyond 512 humans per env:
* the on-device reset (snp_reset) at N up to 4096 against the host generators, and its CTA-per-env kernel against the warp kernel
  bit for bit in every output;
* TiledCrowdEngine.run_checks at any N against LargeCrowd per env and the oracle, and at N <= 512 against CrowdEngine's snp_checks;
* BatchedSocialNavGym on the tiled path: bit for bit a TiledCrowdEngine with spatial_order=False, the same rewards and infos and
  observations in the generator's order with it, restarts of finished envs, and what stays refused."""
import functools

import numpy as np
import pytest
import torch

import oracle
from oracle import OracleConfig
from test_gpu_large_parity import _f32
from test_gpu_reset import _rows

pytestmark = pytest.mark.gpu

DT = 0.0125


# ---------------------------------------------------------------------------------------------------------------- reset
RESET_CASES = [("circle_crossing", False), ("ccso_synthetic", False), ("circle_crossing", True)]


@functools.lru_cache(maxsize=None)
def _host_scenario(name, rand, E, N, R):
    from social_navigation_pyenvs_b200 import scenarios
    if name == "ccso_synthetic":
        return scenarios.ccso_synthetic(E, N, 2000, circle_radius=R)
    return scenarios.circular_crossing(E, N, 2000, circle_radius=R, randomize_attributes=rand)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("N", [600, 1024, 2048, 4096])
@pytest.mark.parametrize("name,rand", RESET_CASES, ids=["cc", "ccso_synthetic", "cc_randattr"])
def test_device_reset_matches_the_host_generators(name, rand, N, dtype):
    """The warp kernel (N <= 1522) and the CTA kernel (above) replay scenarios.py at the same seeds: radii, masses and speeds
    exact, positions, headings and goals up to the last ulp of cos / sin (relative to the circle's radius)."""
    from social_navigation_pyenvs_b200 import TiledCrowdEngine
    E, R = (4 if N <= 1024 else 2), float(N)
    sc = _host_scenario(name, rand, E, N, R)
    eng = TiledCrowdEngine("hsfm_farina", E, N, G=2, dtype=dtype, has_robot=True)
    eng.reset_scenario(name, seed0=2000, circle_radius=R, randomize_attributes=rand)
    rows, goals, cnt = _rows(eng)
    S, G, robot = sc["states"], sc["goals"], sc["robot"]
    if dtype == torch.float32:
        S, G, robot = _f32(S, G, robot)
    tol = 1e-13 * R if dtype == torch.float64 else 1e-6 * R
    assert np.array_equal(rows[..., [8, 9, 12]], S[..., [8, 9, 12]])
    assert np.abs(rows - S).max() <= tol
    assert np.abs(goals - G).max() <= tol and (cnt == 2).all()
    rob, _ = eng.robot_rows()
    assert np.array_equal(rob[:, [0, 1, 8, 10, 11]], robot[:, [0, 1, 8, 10, 11]])


def test_masked_reset_rewrites_only_the_selected_envs():
    """reset with a mask on the CTA kernel: the selected envs equal a full reset with their seeds, the others keep every bit."""
    from social_navigation_pyenvs_b200 import TiledCrowdEngine
    E, N, R = 4, 2048, 2048.0
    eng = TiledCrowdEngine("sfm_guo", E, N, G=2, has_robot=True)
    eng.reset_scenario("circle_crossing", seed0=100, circle_radius=R)
    keep = [t.clone() for t in (eng.dyn, eng.stat, eng.goals, eng.goal_cnt, eng.robot)]
    mask = torch.tensor([True, False, True, False], device=eng.device)
    seeds = np.array([500, 501, 502, 503])
    eng.reset_scenario("circle_crossing", seeds=seeds, mask=mask, circle_radius=R)
    ref = TiledCrowdEngine("sfm_guo", E, N, G=2, has_robot=True)
    ref.reset_scenario("circle_crossing", seeds=seeds, circle_radius=R)
    sel, rest = torch.tensor([0, 2], device=eng.device), torch.tensor([1, 3], device=eng.device)
    for got, old, new in zip((eng.dyn, eng.stat, eng.goals, eng.goal_cnt, eng.robot), keep, (ref.dyn, ref.stat, ref.goals, ref.goal_cnt, ref.robot)):
        axis = -1 if got is eng.robot else -2  # the env axis
        assert torch.equal(got.index_select(axis, sel), new.index_select(axis, sel))
        assert torch.equal(got.index_select(axis, rest), old.index_select(axis, rest))


def _reset_outputs(N, dtype, scenario, rand, force_cta):
    from social_navigation_pyenvs_b200 import TiledCrowdEngine
    E = 8
    eng = TiledCrowdEngine("hsfm_new_guo", E, N, G=2, dtype=dtype, has_robot=True)
    eng.time_now.fill_(3.0)
    eng.flags.fill_(7)
    # parallel traffic: a strip long enough for N humans of radius up to 0.5 (social_nav_sim.py:327-329)
    scen, draws = eng.reset_scenario(scenario, seed0=77, randomize_attributes=rand, circle_radius=max(7.0, float(N)),
                                     traffic_length=max(14.0, 2.0 * N), traffic_height=3.0, force_cta=force_cta)
    return [t.clone() for t in (eng.dyn, eng.stat, eng.goals, eng.goal_idx, eng.goal_cnt, eng.robot, eng.time_now, eng.flags, scen, draws)]


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("N", [5, 25, 300, 1024, 1500])
def test_cta_kernel_equals_the_warp_kernel_bit_for_bit(N, dtype):
    """snp_reset_args bit 0 (SNP_RESET_FORCE_CTA) where the warp kernel fits: every output the same bits, the draw count included."""
    cases = [("circle_crossing", False), ("circle_crossing", True), ("ccso_synthetic", False), ("parallel_traffic", False),
             ("parallel_traffic", True), ("hybrid_scenario", False)] + ([("circular_crossing_with_static_obstacles", False)] if N <= 10 else [])
    for scenario, rand in cases:
        warp = _reset_outputs(N, dtype, scenario, rand, False)
        cta = _reset_outputs(N, dtype, scenario, rand, True)
        for k, (a, b) in enumerate(zip(warp, cta)):
            assert torch.equal(a, b), (scenario, rand, k)
        assert (warp[-1] > 0).all()


# ---------------------------------------------------------------------------------------------------------------- checks
E_CHK = 4


@functools.lru_cache(maxsize=None)
def _check_envs(N):
    """E_CHK crowds of N humans on a jittered grid with random velocities; env 0's robot overlaps a human (collision), env 1's sits
    on its goal, envs 2 and 3 are free and moving through the crowd."""
    rng = np.random.default_rng(N)
    side = int(np.ceil(np.sqrt(N)))
    S = np.zeros((E_CHK, N, 13))
    G = np.zeros((E_CHK, N, 2, 2))
    robots = np.zeros((E_CHK, 13))
    for e in range(E_CHK):
        g = np.stack(np.meshgrid(np.arange(side), np.arange(side), indexing="ij"), -1).reshape(-1, 2)[:N] * 1.1
        S[e, :, 0:2] = g + rng.uniform(-0.1, 0.1, (N, 2))
        S[e, :, 2] = rng.uniform(-np.pi, np.pi, N)
        S[e, :, 3:5] = rng.uniform(-1, 1, (N, 2))
        S[e, :, 5:8] = 0.0
        S[e, :, 8], S[e, :, 9], S[e, :, 12] = 0.3, 75.0, 1.0
        S[e, :, 10:12] = S[e, :, 0:2] + 5.0
        G[e, :, 0] = S[e, :, 10:12]
        G[e, :, 1] = np.nan
        h = S[e, rng.integers(N)]
        pos = {0: h[0:2] + [0.2, 0.1], 1: h[0:2] + [0.55, 0.55], 2: h[0:2] + [0.55, 0.0], 3: h[0:2] + [0.0, 0.55]}[e]
        goal = pos + ([0.1, 0.0] if e == 1 else [3.0, 2.0])
        robots[e, 0:2], robots[e, 2], robots[e, 8], robots[e, 9], robots[e, 10:12], robots[e, 12] = pos, 0.3 * e, 0.3, 80.0, goal, 1.0
    return S, G, robots


def _check_actions(kinematics):
    return np.array([[0.9, 0.4], [0.0, 0.2], [1.0, -0.3], [0.2, 0.9]]) if kinematics == "holonomic" else \
        np.array([[0.9, 0.1], [0.2, 0.0], [1.0, -0.05], [0.6, 0.2]])


def _tiled(model, S, G, robots, dtype, visible):
    from social_navigation_pyenvs_b200 import TiledCrowdEngine
    eng = TiledCrowdEngine.from_reference_arrays(model, S, G, robot=robots, dtype=dtype)
    eng.consider_robot = visible
    return eng


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("visible", [True, False], ids=["visible", "invisible"])
@pytest.mark.parametrize("kinematics", ["holonomic", "unicycle"])
@pytest.mark.parametrize("N", [600, 2048])
def test_tiled_checks_equal_large_crowd_and_the_oracle(N, kinematics, visible, dtype):
    """run_checks (pre and post), collision_detection_and_reaching_goal and check_actual_collisions_and_goal of a batch against a
    LargeCrowd of each env alone bit for bit, and (holonomic) against oracle.checks on the same rows bit for bit."""
    from social_navigation_pyenvs_b200.large import LargeCrowd
    S, G, robots = _check_envs(N)
    act = _check_actions(kinematics)
    if dtype == torch.float32:
        S, G, robots, act = _f32(S, G, robots, act)
    model = "sfm_helbing"  # the stored velocity is the one the checks read
    eng = _tiled(model, S, G, robots, dtype, visible)
    eng.flags.fill_(-1)
    eng.checks.fill_(np.nan)
    f = eng.run_checks(act, pre=True, post=True, kinematics=kinematics)
    mode = 1 if kinematics == "holonomic" else 3
    for e in range(E_CHK):
        one = LargeCrowd(model, S[e], G[e], dtype=dtype, robot=robots[e], consider_robot=visible)
        one.eng.action.copy_(torch.as_tensor(act[e].reshape(2, 1), dtype=dtype))
        one.eng.flags.zero_()
        one.eng.checks.zero_()
        one._checks(DT, mode, pre=True)
        one._checks(DT, mode, pre=False)
        assert int(eng.flags[e]) == int(one.eng.flags[0]) and torch.equal(eng.checks[e], one.eng.checks[0]), e
    assert f["collision"][0] and f["reaching_goal"][1]
    if kinematics == "holonomic":
        consts = np.array(eng.consts)
        ref = oracle.checks(S, N, robots, act, np.zeros(E_CHK), consts)
        assert np.array_equal(f["collision"], ref[:, 0] != 0) and np.array_equal(f["dmin"], ref[:, 1])
        assert np.array_equal(f["reaching_goal"], ref[:, 2] != 0) and np.array_equal(f["reward"], ref[:, 3])
        assert np.array_equal(f["info"], ref[:, 6].astype(int))
        assert np.array_equal(f["actual_collision"], ref[:, 7] != 0) and np.array_equal(f["actual_dmin"], ref[:, 8])
        assert np.array_equal(f["actual_goal"], ref[:, 9] != 0)
        col, dmin, goal = eng.collision_detection_and_reaching_goal(act)
        assert np.array_equal(col, ref[:, 0] != 0) and np.array_equal(dmin, ref[:, 1]) and np.array_equal(goal, ref[:, 2] != 0)
        acol, admin, agoal = eng.check_actual_collisions_and_goal()
        assert np.array_equal(acol, ref[:, 7] != 0) and np.array_equal(admin, ref[:, 8]) and np.array_equal(agoal, ref[:, 9] != 0)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("N", [25, 300, 512])
def test_tiled_checks_up_to_512_humans_are_snp_checks(N, dtype):
    """At N <= 512 TiledCrowdEngine.run_checks is CrowdEngine's (snp_checks): flags and checks [E][4] bit for bit, for a headed
    model too."""
    from social_navigation_pyenvs_b200 import CrowdEngine
    S, G, robots = _check_envs(N)
    act = _check_actions("holonomic")
    if dtype == torch.float32:
        S, G, robots, act = _f32(S, G, robots, act)
    for model in ("sfm_helbing", "hsfm_new_guo"):
        tiled = _tiled(model, S, G, robots, dtype, False)
        fused = CrowdEngine.from_reference_arrays(model, S, G, robot=robots, dtype=dtype)
        for pre, post in ((True, True), (True, False), (False, True)):
            tiled.run_checks(act, pre, post)
            fused.run_checks(act, pre, post)
            assert torch.equal(tiled.flags, fused.flags) and torch.equal(tiled.checks, fused.checks), (model, pre, post)


# ---------------------------------------------------------------------------------------------------------------- gym
E_GYM, N_GYM, R_GYM = 8, 1024, 512.0
GYM_MODEL = "hsfm_new_guo"


def _gym(spatial_order, dtype=torch.float64, **kw):
    from social_navigation_pyenvs_b200 import scenarios
    from social_navigation_pyenvs_b200.social_nav_gym import BatchedSocialNavGym
    g = BatchedSocialNavGym(E_GYM, dtype=dtype)
    g.configure(dict(human_policy=GYM_MODEL, human_num=N_GYM, circle_radius=R_GYM, robot_visible=True, spatial_order=spatial_order,
                     walls=scenarios.pack_walls(scenarios.EXAMPLE_WALLS), **kw))
    return g


def _gym_actions(t):
    return np.stack([np.full(E_GYM, 0.3 * np.sin(0.3 * t)), np.linspace(0.5, 1.0, E_GYM)], 1)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
def test_gym_without_spatial_order_is_the_tiled_engine_bit_for_bit(dtype):
    from social_navigation_pyenvs_b200 import TiledCrowdEngine, scenarios
    g = _gym(False, dtype)
    obs, _ = g.reset("train", test_case=0, on_device=False)
    assert isinstance(g.engine, TiledCrowdEngine)
    sc = scenarios.circular_crossing(E_GYM, N_GYM, 2000 + np.arange(E_GYM), R_GYM)
    robot = sc["robot"].copy()
    robot[:, 3:5] = 0.0
    ref = TiledCrowdEngine.from_reference_arrays(GYM_MODEL, np.concatenate([sc["states"], robot[:, None]], 1), sc["goals"],
                                                 walls=g.walls, consider_robot=True, dtype=dtype)
    ref.consts = list(g.engine.consts)
    from social_navigation_pyenvs_b200 import _lib as L
    cols = lambda e: torch.stack([e.dyn[L.DYN_PX], e.dyn[L.DYN_PY], e.dyn[L.DYN_VX], e.dyn[L.DYN_VY], e.stat[L.STAT_R]], -1).double().cpu().numpy()
    assert np.array_equal(obs, cols(ref))
    for t in range(20):
        o, r, term, trunc, info = g.step(_gym_actions(t))
        ref.step(_gym_actions(t), g.time_step, n_substeps=g.time_step_factor, pre_checks=True)
        f = ref.decode_flags()
        assert np.array_equal(o, cols(ref)), t
        assert np.array_equal(r, f["reward"]) and np.array_equal(info, f["info"]), t
        assert np.array_equal(term, f["terminated"]) and np.array_equal(trunc, f["truncated"]), t


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
def test_gym_with_spatial_order_matches_the_oracle_in_generator_order(dtype):
    """Device reset, one sub-step per gym step (robot_time_step = time_step): the first step against the oracle within the parity
    tolerance, in the generator's order; 20 steps against the gym without spatial_order: observations within the tolerance, reward,
    terminated, truncated and info the same."""
    from social_navigation_pyenvs_b200 import scenarios
    a, b = _gym(False, dtype, robot_time_step=DT), _gym(True, dtype, robot_time_step=DT)
    oa, _ = a.reset("train", test_case=0)
    ob, _ = b.reset("train", test_case=0)
    assert np.array_equal(oa, ob)
    assert not np.array_equal(b.engine.dyn[0].cpu().numpy(), a.engine.dyn[0].cpu().numpy())  # b's rows are re-numbered
    tol = 1e-9 if dtype == torch.float64 else 1e-4
    sc = scenarios.circular_crossing(E_GYM, N_GYM, 2000 + np.arange(E_GYM), R_GYM)
    S = np.concatenate([sc["states"], sc["robot"][:, None]], 1)
    S[:, N_GYM, 3:8] = 0.0  # the robot at rest (social_nav_gym.py:213)
    goals, act = sc["goals"], _gym_actions(0)
    if dtype == torch.float32:
        S, goals, act = _f32(S, goals, act)
    cfg = OracleConfig(oracle.type_code(GYM_MODEL), True, True, False)
    walls = b.walls
    ref, _, _ = oracle.update_humans(cfg, S, goals, walls, np.tile(oracle.default_params(GYM_MODEL), (E_GYM, N_GYM, 1)),
                                     np.zeros((E_GYM, N_GYM + 1)), np.zeros((E_GYM, N_GYM, 2)), DT, b.time_step_factor,
                                     robot_vel=act, n_threads=8)
    chk = oracle.checks(S, N_GYM, S[:, N_GYM], act, np.zeros(E_GYM), np.array(b.engine.consts))
    for t in range(20):
        ra, rb = a.step(_gym_actions(t)), b.step(_gym_actions(t))
        scale = np.maximum(np.abs(ra[0]), 1.0)
        assert (np.abs(rb[0] - ra[0]) / scale).max() <= tol, t
        for k in range(1, 5):
            assert np.array_equal(ra[k], rb[k]), (t, k)
        if t == 0:
            want = ref[:, :N_GYM][..., [0, 1, 3, 4, 8]]
            assert (np.abs(rb[0] - want) / np.maximum(np.abs(want), 1.0)).max() <= tol
            assert np.array_equal(rb[1], chk[:, 3]) and np.array_equal(rb[4], chk[:, 6].astype(int))


def test_gym_restarts_finished_envs_and_steps_on():
    """reset_finished on the tiled path: the restarted envs show the next cases in the generator's order, the others keep every
    bit of their observation (re-numbering only permutes rows), and the gym steps on."""
    b = _gym(True)
    b.reset("train", test_case=0)
    for t in range(2):
        b.step(_gym_actions(t))
    before = b.observation()
    fin = np.zeros(E_GYM, bool)
    fin[[1, 6]] = True
    after = b.reset_finished(fin, "train")
    assert np.array_equal(after[~fin], before[~fin])
    from social_navigation_pyenvs_b200.social_nav_gym import BatchedSocialNavGym
    ref = BatchedSocialNavGym(2)
    ref.configure(dict(human_policy=GYM_MODEL, human_num=N_GYM, circle_radius=R_GYM, robot_visible=True, walls=b.walls))
    obs_ref, _ = ref.reset("train", test_case=E_GYM)
    assert np.array_equal(after[fin], obs_ref)
    o, r, term, trunc, info = b.step(_gym_actions(2))
    assert np.isfinite(o).all() and np.isfinite(r).all()


def test_gym_refuses_what_the_tiled_path_lacks():
    from social_navigation_pyenvs_b200.social_nav_gym import BatchedSocialNavGym
    g = BatchedSocialNavGym(2)
    g.configure(dict(human_policy="sfm_helbing", human_num=600, train_val_sim="parallel_traffic", traffic_length=600.0, traffic_height=3.0))
    g.reset("train", test_case=0)
    with pytest.raises(NotImplementedError):
        g.step(np.zeros((2, 2)))
    c = _gym(True)
    c.reset("train", test_case=0)
    c.set_robot_motion_model("sfm_helbing")
    with pytest.raises(NotImplementedError):
        c.imitation_learning_step()
