"""CADRL's action choice on the device (snp_value_lookahead through CrowdEngine / TiledCrowdEngine.predict and predict_from) against
its restatement in PyTorch: the lookahead's rotated rows rounded to fp32, the same nn.Sequential, the minimum over the humans, then
reward + gamma ** (dt * v_pref) * minimum and the first argmax -- for both crowd dtypes, 13 and 15 values per row, the peek and the
constant-velocity propagation, N from 1 to 4096 (whole envs and envs split over CTAs) and 81 or 7 actions."""
import numpy as np
import pytest
import torch

from oracle import reference
from test_gpu_block_packed import _look_batch
from test_gpu_lookahead import _actions

pytestmark = pytest.mark.gpu

DT, GAMMA = 0.25, 0.9
NS = [1, 5, 25, 33, 512, 700, 4096]


def _net(visible, seed=7, widths=(150, 100, 100)):
    torch.manual_seed(seed)
    dims = [15 if visible else 13, *widths, 1]
    layers = []
    for i in range(len(dims) - 1):
        layers.append(torch.nn.Linear(dims[i], dims[i + 1]))
        if i + 2 < len(dims):
            layers.append(torch.nn.ReLU())
    return torch.nn.Sequential(*layers).cuda()


def _engine(N, dtype, model="hsfm_farina", seed=11, tiled=None):
    from social_navigation_pyenvs_b200 import CrowdEngine, TiledCrowdEngine
    E = 13 if N <= 33 else (5 if N <= 700 else 3)  # 2025 pairs of an env with 81 actions and 25 humans: the last warp group is ragged
    S, G, R = _look_batch(E, N, seed + N)
    R[2::5, 10:12] = R[2::5, 0:2] + [0.1, -0.2]  # robots within their radius of the goal: predict's zero action
    cls = (TiledCrowdEngine if N > 512 else CrowdEngine) if tiled is None else (TiledCrowdEngine if tiled else CrowdEngine)
    return cls.from_reference_arrays(model, S, G, consider_robot=False, all_params_equal=True, robot=R, dtype=dtype)


def _torch_choice(eng, net, nxt, visible, yaw_from_next):
    """The restatement: lookahead_from rows .float() -> net -> min over humans -> reward + gamma ** (dt v_pref) * m.double()."""
    from social_navigation_pyenvs_b200 import _lib as L
    rot, rew = eng.lookahead_from(nxt, DT, theta_and_omega_visible=visible, yaw_from_next=yaw_from_next)
    with torch.no_grad():
        m = torch.cat([net(rot[i:i + 1].float()).squeeze(-1).amin(-1) for i in range(eng.E)])
    disc = GAMMA ** (DT * eng.robot[L.ROBOT_VD].double())
    return m, rew.clone(), rew + disc[:, None] * m.double(), disc


def _check_choice(best, values, m_fused, m_t, v_t):
    assert ((m_fused - m_t.double()).abs() <= 1e-5 * m_t.double().abs().clamp(min=1)).all()
    top2 = v_t.topk(2, dim=1).values if v_t.shape[1] > 1 else torch.cat([v_t, v_t - 1], 1)
    gap = top2[:, 0] - top2[:, 1]
    clear = gap > 2e-5 * top2[:, 0].abs().clamp(min=1)
    first = v_t.argmax(1)  # torch returns the first index of the maximum
    assert torch.equal(best[clear], first[clear])
    picked = v_t.gather(1, best[:, None])[:, 0]
    assert (top2[:, 0] - picked <= 2e-5 * top2[:, 0].abs().clamp(min=1) + gap)[~clear].all()
    assert torch.equal(values.argmax(1), best)  # the returned values agree with the returned choice


@pytest.mark.parametrize("A", [81, 7])
@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("visible", [False, True])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_predict_against_torch(dtype, visible, N, A):
    from social_navigation_pyenvs_b200 import TiledCrowdEngine, _lib as L
    eng = _engine(N, dtype)
    eng.set_action_space(_actions()[:A] if A == 81 else _actions()[::12][:A])
    net = _net(visible)
    eng.set_value_network(net, GAMMA)
    modes = [False] if isinstance(eng, TiledCrowdEngine) else [True, False]
    for query_env in modes:
        before = (eng.dyn[:L.DYN_DFX].clone(), eng.goal_idx.clone(), eng.robot.clone())
        best, values, reached = (t.clone() for t in eng.predict(DT, theta_and_omega_visible=visible, query_env=query_env))
        assert torch.equal(eng.dyn[:L.DYN_DFX], before[0]) and torch.equal(eng.goal_idx, before[1]) and torch.equal(eng.robot, before[2])
        nxt = eng._peek_buf.clone()
        assert best.dtype == torch.int64 and values.dtype == torch.float64 and reached.dtype == torch.bool
        m_t, rew, v_t, disc = _torch_choice(eng, net, nxt, visible, yaw_from_next=not query_env)
        m_fused = (values - rew) / disc[:, None]
        _check_choice(best, values, m_fused, m_t, v_t)
        r = eng.robot.double()
        dx, dy = r[L.ROBOT_PX] - r[L.ROBOT_GX], r[L.ROBOT_PY] - r[L.ROBOT_GY]
        assert torch.equal(reached, torch.sqrt(dx * dx + dy * dy) < r[L.ROBOT_R]) and reached.any() and not reached.all()
        # the same bits from predict_from on the same `next`, and with every env's humans split over CTAs in chunks of 32
        for split in (False, True):
            b2, v2, r2 = eng.predict_from(nxt, DT, theta_and_omega_visible=visible, yaw_from_next=not query_env, split_humans=split)
            assert torch.equal(b2, best) and torch.equal(v2, values) and torch.equal(r2, reached), (query_env, split)


@pytest.mark.parametrize("N", [25, 700])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_zero_network_leaves_the_lookahead_rewards(dtype, N):
    """With every weight zeroed the minimum is 0 and values are the lookahead's rewards bit for bit; the scenes hold every kind of
    reward (collision, goal, discomfort, nothing), some robots sit on their goal."""
    eng = _engine(N, dtype)
    eng.set_action_space(_actions())
    net = _net(False)
    with torch.no_grad():
        for p in net.parameters():
            p.zero_()
    eng.set_value_network(net, GAMMA)
    nxt = eng.constant_velocity_next(DT)
    for split in (False, True):
        best, values, reached = eng.predict_from(nxt, DT, yaw_from_next=True, split_humans=split)
        _, rew = eng.lookahead_from(nxt, DT, yaw_from_next=True)
        assert torch.equal(values, rew), split
        assert torch.equal(best, rew.argmax(1))
    kinds = {(rew == -0.25).any().item(), (rew == 1.0).any().item(), ((rew < 0) & (rew > -0.25)).any().item(), (rew == 0).any().item()}
    assert kinds == {True}


@pytest.mark.parametrize("N", [5, 33, 512])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_crowd_and_tiled_engines_choose_alike(dtype, N):
    """Built from the same rows, CrowdEngine and TiledCrowdEngine give the same values and choices bit for bit (query_env=False)."""
    from social_navigation_pyenvs_b200 import TiledCrowdEngine
    out = []
    for tiled in (False, True):
        eng = _engine(N, dtype, model="sfm_guo", tiled=tiled)
        assert isinstance(eng, TiledCrowdEngine) == tiled
        eng.set_action_space(_actions())
        eng.set_value_network(_net(True, seed=3, widths=(64, 40)), GAMMA)
        out.append([t.clone() for t in eng.predict(DT, theta_and_omega_visible=True, query_env=False)])
    for a, b in zip(*out):
        assert torch.equal(a, b)


@pytest.mark.parametrize("N", [25, 700])
@pytest.mark.parametrize("visible", [False, True])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_fused_rows_are_the_lookahead_rows_bit_for_bit(dtype, visible, N):
    """A one-hot Linear(13 | 15, 1) without bias outputs one column of the row exactly, so with gamma = 1 the values are
    reward + min over the humans of that column of the fused row: equal, bit for bit, to the same expression on the lookahead's rows
    rounded to fp32 -- for every column, whole-env and split."""
    eng = _engine(N, dtype)
    eng.set_action_space(_actions())
    ow = 15 if visible else 13
    nxt = eng.constant_velocity_next(DT).clone()
    rot, rew = eng.lookahead_from(nxt, DT, theta_and_omega_visible=visible, yaw_from_next=True)
    rows, rew = rot.float(), rew.clone()
    for c in range(ow):
        net = torch.nn.Linear(ow, 1, bias=False).cuda()
        with torch.no_grad():
            net.weight.zero_()
            net.weight[0, c] = 1.0
        eng.set_value_network(net, 1.0)
        want = rew + rows[..., c].amin(-1).double()
        for split in (False, True):
            _, values, _ = eng.predict_from(nxt, DT, theta_and_omega_visible=visible, yaw_from_next=True, split_humans=split)
            assert torch.equal(values, want), (c, split)


def test_tiled_engine_predict_with_a_query_raises():
    """The tiled path has no peek: predict(query_env=True) raises as lookahead(query_env=True) does."""
    eng = _engine(700, torch.float64)
    eng.set_action_space(_actions())
    eng.set_value_network(_net(False), GAMMA)
    with pytest.raises(NotImplementedError, match="TiledCrowdEngine"):
        eng.predict(DT, query_env=True)


def test_predict_refuses_a_mismatched_input_width():
    eng = _engine(5, torch.float64)
    eng.set_action_space(_actions())
    eng.set_value_network(_net(True), GAMMA)
    with pytest.raises(ValueError, match="snp_value_lookahead"):
        eng.predict(DT, theta_and_omega_visible=False, query_env=False)


@pytest.mark.skipif(not reference.available(), reason="live reference not staged (oracle/build.py)")
@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_the_reference_cadrl_chooses_the_same_action(seed):
    """The reference's own CADRL (crowd_nav/policy/cadrl.py, configured from its policy.config, phase 'test', query_env False) and
    predict() on a 5-human env, against the engine's predict(query_env=False) with the same ValueNetwork object: the same action."""
    import configparser
    import os
    reference.install()
    from crowd_nav.policy.cadrl import CADRL
    from crowd_nav.utils.state import FullState, JointState, ObservableState
    from social_navigation_pyenvs_b200 import CrowdEngine
    policy = CADRL()
    cfg = configparser.RawConfigParser()
    cfg.read(os.path.join(reference.root(), "crowd_nav", "configs", "policy.config"))
    policy.configure(cfg)
    policy.set_phase("test")
    policy.set_device(torch.device("cpu"))
    policy.time_step, policy.query_env = DT, False
    S, G, R = _look_batch(1, 5, 300 + seed)
    eng = CrowdEngine.from_reference_arrays("sfm_helbing", S, G, consider_robot=False, all_params_equal=True, robot=R)
    eng.set_action_space(_actions())
    eng.set_value_network(policy.model, policy.gamma)
    best, _, reached = eng.predict(DT, query_env=False)
    r = R[0]
    state = JointState(FullState(r[0], r[1], r[3], r[4], r[8], r[10], r[11], r[12], r[2]),
                       [ObservableState(h[0], h[1], h[3], h[4], h[8]) for h in S[0]])
    with torch.no_grad():
        action = policy.predict(state)
    want = np.zeros(2) if bool(reached[0]) else _actions()[int(best[0])]
    assert np.allclose([action.vx, action.vy], want, atol=1e-9), (action, want)
