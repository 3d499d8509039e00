"""Re-numbering a crowd patch by patch on the device mid-run (LargeCrowd.renumber, TiledCrowdEngine.renumber):

* the device permutation is scenarios.spatial_order element for element (rounding and np.array_split edges of the strip count,
  exact ties in x and y, -0.0 against +0.0, fp32 positions, deal_tiles at 2 and 8 ranks), and a NaN position raises;
* after renumber() every per-agent array is the old one indexed by perm, bit for bit -- dyn with the carried desired force, stat,
  goals, goal_idx after goal switches, goal_cnt -- and so are the radii; the view equals that of a crowd loaded with the permuted
  arrays and the tile boxes are those of the view;
* a crowd stepped, re-numbered and stepped again equals a crowd loaded with the permuted arrays and stepped the same way, bit for bit
  (state, robot, flags, checks, clock, laser ranges and hit indices), with culling on and off and with unit_capacity="auto", over
  the fused one-call loop and one call per sub-step; un-permuted it is the oracle's one sub-step from the re-numbered state;
* env e of a TiledCrowdEngine after renumber() and a step equals a LargeCrowd of env e alone re-numbered and stepped.
Sharded crowds: tests/test_gpu_multi_renumber.py."""
import functools

import numpy as np
import pytest
import torch

import oracle
from oracle import OracleConfig
from helpers import rotate_goals_to
from test_gpu_large_parity import _crowd_with_walls, _err, _f32, _poison
from test_gpu_large_robot import _robot_row

pytestmark = pytest.mark.gpu

DT = 0.0125
ROBOT_SAFETY = 0.05
ACTION = np.array([0.9, 0.35])
DTYPES = pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])


def _device_order(pos, dtype, world=1):
    from social_navigation_pyenvs_b200.large import device_spatial_order
    t = torch.as_tensor(np.ascontiguousarray(pos.T), dtype=dtype, device="cuda")
    return device_spatial_order(t[0], t[1], world=world).cpu().numpy()


# ---- the permutation ----

@DTYPES
@pytest.mark.parametrize("n", [64, 513, 576, 1000, 1600, 5184])
def test_device_order_is_spatial_order(n, dtype):
    from social_navigation_pyenvs_b200 import scenarios
    pos = np.random.RandomState(n).uniform(-40.0, 40.0, (n, 2))
    if dtype == torch.float32:
        pos = pos.astype(np.float32).astype(np.float64)  # what the fp32 crowd holds, as NumPy sees it widened
    assert np.array_equal(_device_order(pos, dtype), scenarios.spatial_order(pos))


@DTYPES
def test_exact_ties_and_signed_zeros_keep_numpy_order(dtype):
    from social_navigation_pyenvs_b200 import scenarios
    rng = np.random.RandomState(5)
    ix, iy = np.meshgrid(np.arange(24), np.arange(24), indexing="ij")
    grid = np.stack([ix.ravel() - 12.0, iy.ravel() - 12.0], 1)[rng.permutation(576)]  # unjittered: exact ties in x and in y
    assert np.array_equal(_device_order(grid, dtype), scenarios.spatial_order(grid))
    zeros = rng.choice([-0.0, 0.0, 1.0, -1.0], (700, 2))  # -0.0 and +0.0 are the same key
    assert (np.signbit(zeros) & (zeros == 0)).any() and (~np.signbit(zeros) & (zeros == 0)).any()
    assert np.array_equal(_device_order(zeros, dtype), scenarios.spatial_order(zeros))


@DTYPES
@pytest.mark.parametrize("world", [2, 8])
def test_tiles_dealt_to_ranks_as_deal_tiles(world, dtype):
    from social_navigation_pyenvs_b200 import scenarios
    for n in (1024, 5120, 65536):
        pos = np.random.RandomState(n + world).uniform(-60.0, 60.0, (n, 2))
        if dtype == torch.float32:
            pos = pos.astype(np.float32).astype(np.float64)
        assert np.array_equal(_device_order(pos, dtype, world), scenarios.deal_tiles(scenarios.spatial_order(pos), world)), n


@DTYPES
def test_batched_envs_are_ordered_each_on_its_own(dtype):
    from social_navigation_pyenvs_b200 import scenarios
    from social_navigation_pyenvs_b200.large import device_spatial_order
    pos = np.random.RandomState(9).uniform(-20.0, 20.0, (3, 1000, 2))
    pos[1] = pos[0]  # two envs with the same humans: each is numbered within itself
    t = torch.as_tensor(pos, dtype=dtype, device="cuda")
    got = device_spatial_order(t[..., 0], t[..., 1]).cpu().numpy()
    for e in range(3):
        assert np.array_equal(got[e], scenarios.spatial_order(t[e].double().cpu().numpy())), e


@DTYPES
def test_non_finite_positions_raise(dtype):
    pos = np.random.RandomState(3).uniform(-5.0, 5.0, (300, 2))
    for bad in (np.nan, np.inf):
        p = pos.copy()
        p[17, 1] = bad
        with pytest.raises(ValueError, match="NaN or infinite"):
            _device_order(p, dtype)


# ---- LargeCrowd ----

@functools.lru_cache(maxsize=None)
def _scene(n, dtype):
    """n humans of the moving ~1500-human crowd with goal switches and per-human safety (some with a one-goal list), the example walls
    and a visible robot near the centre.  n = 1024: whole tiles (one C call per step); 1000: a ragged last tile (one per sub-step)."""
    from social_navigation_pyenvs_b200 import scenarios
    S, G, saf = _crowd_with_walls(scenarios.EXAMPLE_WALLS, 0.7, seed=21)
    S, G, saf = S[:n].copy(), G[:n].copy(), saf[:n].copy()
    G[::7, 1] = np.nan
    walls, robot = scenarios.pack_walls(scenarios.EXAMPLE_WALLS), _robot_row(S)
    if dtype == torch.float32:
        S, G, saf, walls, robot = _f32(S, G, saf, walls, robot)
    return S, G, saf, walls, robot


def _large(model, scene, dtype, unit_capacity=None, culling=True):
    from social_navigation_pyenvs_b200.large import LargeCrowd
    S, G, saf, walls, robot = scene
    c = LargeCrowd(model, S, G, walls=walls, safety=saf, dtype=dtype, robot=robot, robot_safety=ROBOT_SAFETY, consider_robot=True,
                   unit_capacity=unit_capacity)
    c.culling = culling
    return c


def _arrays(crowd):
    e = crowd.eng
    return [t.cpu().numpy().copy() for t in (e.dyn, e.stat, e.goals, e.goal_idx, e.goal_cnt, crowd.radius)]


def _loaded(model, scene, dtype, arrays, robot_from, **kw):
    """A crowd built from the scene, then loaded with `arrays` (those of _arrays) and the robot and clock of `robot_from`, its view
    published from them."""
    c = _large(model, scene, dtype, **kw)
    e, src = c.eng, [torch.as_tensor(a, device="cuda") for a in arrays]
    for t, a in zip((e.dyn, e.stat, e.goals, e.goal_idx, e.goal_cnt, c.radius), src):
        t.copy_(a)
    e.robot.copy_(robot_from.eng.robot)
    e.time_now.copy_(robot_from.eng.time_now)
    c._publish()
    return c


def _permuted(arrays, perm):
    return [a[..., perm] for a in arrays]


def _gym_step(crowd, k):
    _poison(crowd, True)
    crowd.step(DT, n_substeps=k, action=ACTION, pre_checks=True, post_checks=True)


def _results(crowd):
    e = crowd.eng
    ranges, hits = crowd.scan(2 * np.pi, 360, 10.0, robot_radius=0.3)
    return ([t.cpu().numpy() for t in (e.dyn, e.goal_idx, e.robot, e.flags, e.checks, e.time_now)] +
            [ranges.cpu().numpy(), hits.cpu().numpy()])


def _boxes(view, M):
    v = view.cpu().numpy()
    T = -(-M // 128)
    pad = lambda row, fill: np.concatenate([row, np.full(T * 128 - M, fill, row.dtype)]).reshape(T, 128)
    x, y, rs = v[0], v[1], v[4]
    return np.stack([pad(x, np.inf).min(1), pad(x, -np.inf).max(1), pad(y, np.inf).min(1), pad(y, -np.inf).max(1), pad(rs, 0).max(1)], 1)


@DTYPES
@pytest.mark.parametrize("n", [1024, 1000])
def test_renumber_moves_every_array_with_its_human(n, dtype):
    from social_navigation_pyenvs_b200 import scenarios
    scene = _scene(n, dtype)
    crowd = _large("hsfm_farina", scene, dtype)
    assert crowd.exchange == ("fused" if n == 1024 else "nccl")
    _gym_step(crowd, 20)
    before = _arrays(crowd)
    assert len(np.unique(before[3])) == 2 and len(np.unique(before[4])) == 2  # goal switches happened, one- and two-goal lists
    assert np.any(before[0][8:10] != 0)  # a carried desired force
    pos = crowd.view[crowd.cur][0:2].double().cpu().numpy().T
    perm = crowd.renumber()
    assert perm.dtype == np.int64 and np.array_equal(perm, scenarios.spatial_order(pos))
    assert not np.array_equal(perm, np.arange(n))
    for a, b in zip(_arrays(crowd), _permuted(before, perm)):  # bit patterns: the unused goal slots are NaN
        assert a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()
    ref = _loaded("hsfm_farina", scene, dtype, _permuted(before, perm), crowd)
    M = crowd.n_total
    assert torch.equal(crowd.view[crowd.cur], ref.view[ref.cur])
    got_boxes = crowd._vbuf[crowd.cur][5 * M:].view(-1, 5).cpu().numpy()
    assert np.array_equal(got_boxes, _boxes(ref.view[ref.cur], M))


@DTYPES
@pytest.mark.parametrize("n,cap,culling", [(1024, None, True), (1024, None, False), (1024, "auto", True), (1000, None, True)],
                         ids=["fused", "no_culling", "auto_units", "per_substep"])
def test_stepping_after_renumber_equals_the_permuted_crowd(n, cap, culling, dtype):
    scene = _scene(n, dtype)
    crowd = _large("sfm_guo", scene, dtype, unit_capacity=cap, culling=culling)
    _gym_step(crowd, 20)
    before = _arrays(crowd)
    perm = crowd.renumber()
    ref = _loaded("sfm_guo", scene, dtype, _permuted(before, perm), crowd, unit_capacity=cap, culling=culling)
    for k in (20, 7):
        _gym_step(crowd, k)
        _gym_step(ref, k)
        for a, b in zip(_results(crowd), _results(ref)):
            assert np.array_equal(a, b)
        if cap == "auto":  # the same units in reach (the capacity differs: the re-numbered crowd grew it before)
            assert crowd.unit_stats()["max_listed"] == ref.unit_stats()["max_listed"]
    assert crowd.decode_flags()["dmin"][0] < 10.0  # the robot sees humans


@DTYPES
def test_renumbered_crowd_against_the_oracle(dtype):
    """One sub-step from the re-numbered state, un-permuted, against oracle.update_humans from the same state in the old numbering
    (desired force carried, goal lists rotated to the current goal, the robot as row n with its holonomic action)."""
    model = "hsfm_farina"
    S, G, saf, walls, robot = scene = _scene(1024, dtype)
    crowd = _large(model, scene, dtype)
    _gym_step(crowd, 20)
    rows = crowd.local_rows(S)
    D = crowd.eng.desired_force()[0]
    Gr = rotate_goals_to(G, rows[:, 10:12])
    n = rows.shape[0]
    start = np.concatenate([rows, crowd.robot_rows()[None]])[None]
    cfg = OracleConfig(oracle.type_code(model), True, True, False)
    ref, _, _ = oracle.update_humans(cfg, start, Gr[None], walls, np.tile(oracle.default_params(model), (1, n, 1)),
                                     np.concatenate([saf, [ROBOT_SAFETY]])[None], D[None], DT, 1, robot_vel=ACTION[None], n_threads=8)
    perm = crowd.renumber()
    crowd.step(DT, n_substeps=1, action=ACTION)
    got = crowd.local_rows(S[perm])[np.argsort(perm)]
    assert _err(got, ref[0, :n]) < (1e-9 if dtype == torch.float64 else 1e-4)


# ---- TiledCrowdEngine ----

@DTYPES
@pytest.mark.parametrize("N", [513, 1000])
def test_every_env_of_a_renumbered_batch_equals_its_own_renumbered_large_crowd(N, dtype):
    from social_navigation_pyenvs_b200 import TiledCrowdEngine, scenarios
    from social_navigation_pyenvs_b200.large import LargeCrowd
    E, model = 3, "hsfm_new_guo"
    scenes = [_crowd_with_walls(scenarios.EXAMPLE_WALLS, 0.7, seed=31 + e) for e in range(E)]
    S, G, saf = (np.stack([s[i][:N] for s in scenes]) for i in range(3))
    walls = scenarios.pack_walls(scenarios.EXAMPLE_WALLS)
    robots = np.stack([_robot_row(S[e], yaw=0.3 * e) for e in range(E)])
    act = np.array([[0.9 - 0.2 * e, 0.35] for e in range(E)])
    if dtype == torch.float32:
        S, G, saf, walls, robots, act = _f32(S, G, saf, walls, robots, act)
    batch = TiledCrowdEngine.from_reference_arrays(model, S, G, walls=walls, safety=saf, robot=robots, dtype=dtype)
    batch.set_robot_rows(robots, safety=np.full(E, ROBOT_SAFETY))
    batch.consider_robot = True
    singles = [LargeCrowd(model, S[e], G[e], walls=walls, safety=saf[e], dtype=dtype, robot=robots[e], robot_safety=ROBOT_SAFETY,
                          consider_robot=True) for e in range(E)]

    def step_all(k):
        batch.scratch.fill_(0xFF)
        batch.step(act, DT, n_substeps=k, pre_checks=True, post_checks=True)
        for e, one in enumerate(singles):
            _poison(one, True)
            one._publish()  # a batch call publishes the view from the state, as a LargeCrowd built from it does
            one.step(DT, n_substeps=k, action=act[e], pre_checks=True, post_checks=True)

    step_all(20)
    pos = torch.stack([batch.dyn[0], batch.dyn[1]], -1).double().cpu().numpy()
    perm = batch.renumber()
    assert perm.shape == (E, N) and perm.dtype == np.int64
    for e, one in enumerate(singles):
        assert np.array_equal(perm[e], scenarios.spatial_order(pos[e])), e
        assert np.array_equal(one.renumber(), perm[e]), e
    step_all(5)
    Sp = np.stack([S[e][perm[e]] for e in range(E)])
    rows, (rob, _) = batch.rows(Sp), batch.robot_rows()
    flags, checks, clock = batch.flags.cpu().numpy(), batch.checks.cpu().numpy(), batch.time_now.cpu().numpy()
    for e, one in enumerate(singles):
        assert np.array_equal(rows[e], one.local_rows(Sp[e])), e
        assert np.array_equal(batch.goal_idx[e].cpu().numpy(), one.eng.goal_idx[0].cpu().numpy()), e
        assert np.array_equal(rob[e], one.robot_rows()), e
        assert flags[e] == int(one.eng.flags[0]) and np.array_equal(checks[e], one.eng.checks[0].cpu().numpy()), e
        assert clock[e] == float(one.eng.time_now[0]), e
