"""The block-packed mapping of the fused step (snp::k_step with CTA = true, 33 <= N <= 512 humans per env) against the oracle.

floor(128/N) env groups share a 128-thread CTA up to N = 128 (groups straddle warp boundaries, the last CTA of a batch may be
partly empty); above that one env runs on a CTA of ceil(N/32)*32 threads.  Reductions (pre-step swept check, post-step admin
min, touch flag, the robot_mode 2 force sum) go through shared memory, the halved pair loop exchanges forces through
[rounds][gpb*N] planes and falls back to the j-ascending loop when those would exceed 64 KiB (fp64 from N = 92, fp32 from N = 129).

Bars (DESIGN section 2): fp64 1e-9 after 20 fused sub-steps, current goals exact, desired force at scale 100; fp32 1e-4 after ONE
sub-step from fp32-rounded inputs (the 20-sub-step fp32 run asserts finiteness and the checks); flags, dmin, reward bit for bit.
Every multi-sub-step fp64 case first shows that its crowd is well conditioned: the oracle run from positions perturbed by 2e-16
(relative) stays within 1e-11 of the unperturbed run, so a failure at 1e-9 points at the kernel, not at the crowd.
"""
import os

import numpy as np
import pytest
import torch

import oracle
from oracle import OracleConfig
from helpers import rel_err, wrap_angle_cols, unicycle_step
from test_gpu_sizes_large import _random_crowd
from test_gpu_lookahead import _actions, _oracle_inputs

pytestmark = pytest.mark.gpu

DT, K = 0.0125, 20
THREADS = os.cpu_count() or 1
MODELS = ["sfm_helbing", "sfm_guo", "sfm_moussaid", "hsfm_farina", "hsfm_guo", "hsfm_moussaid", "hsfm_new", "hsfm_new_guo", "hsfm_new_moussaid"]
# N of the shape table: first N of the mapping (3 groups on 99 of 128 threads), largest N with 3 groups, odd N with 2 groups, even
# N with the antipodal pair on a full CTA, one env per CTA, last / first fp64 N of the halved loop (91: 65,520 B of planes; 92:
# ordered), last fp32 N of the halved loop and last N on 128 threads, first N above 128 threads (one live lane in the last warp),
# whole warps vs a ragged last warp, odd and even at the limit
SHAPES = [33, 42, 43, 64, 65, 91, 92, 128, 129, 256, 257, 511, 512]
DTYPES = [pytest.param(torch.float64, id="f64"), pytest.param(torch.float32, id="f32")]
ERRS = {}  # (section, dtype) -> largest error seen; printed at the end of the module (pytest -s)


@pytest.fixture(scope="module", autouse=True)
def _error_report():
    yield
    for (section, dt), e in sorted(ERRS.items()):
        print(f"[block-packed] {section:<12} {dt}: largest error {e:.3e}")


def _record(section, dtype, err):
    key = (section, "f64" if dtype == torch.float64 else "f32")
    ERRS[key] = max(ERRS.get(key, 0.0), float(err))


def _gpb(N):
    return 128 // N if N <= 128 else 1


def _envs(N):
    """E that spans several CTAs without being a multiple of the groups per CTA: the last CTA is partly empty."""
    return {3: 7, 2: 5}.get(_gpb(N), 3)


def _f32(*arrays):
    return [None if a is None else np.asarray(a, np.float64).astype(np.float32).astype(np.float64) for a in arrays]


def _state_err(got, ref):
    """Largest relative error of human rows [..., :8] with the heading compared as an angle."""
    return float(rel_err(wrap_angle_cols(got[..., :8], ref[..., :8]), ref[..., :8]).max())


def _clear_cells(S, spread, k):
    """Centres of the k grid cells of the crowd's interior farthest from every human of every env (robot / obstacle sites)."""
    side = int(np.ceil(np.sqrt(S.shape[1])))
    rows = (S.shape[1] + side - 1) // side  # grid rows that hold humans (filled column by column)
    cand = np.array([[(a + 0.5) * spread, (b + 0.5) * spread] for a in range(max(rows - 1, 1)) for b in range(side - 1)])
    clear = np.array([(np.linalg.norm(S[:, :, 0:2] - c, axis=-1) - S[:, :, 8]).min() for c in cand])
    order = np.argsort(-clear)
    return cand[order[:k]], clear[order[:k]]


def _walls(S, spread, inner_site, per_env_shift=None):
    """scenarios.EXAMPLE_WALLS moved against the crowd's right edge, plus a small triangle inside the crowd at `inner_site`."""
    from social_navigation_pyenvs_b200 import scenarios
    xmax = S[:, :, 0].max() + S[:, :, 8].max()
    ymid = 0.5 * (S[:, :, 1].min() + S[:, :, 1].max())
    shift = np.array([xmax + 0.6 + 7.0, ymid + 3.0])
    polys = [[[x + shift[0], y + shift[1]] for x, y in p] for p in scenarios.EXAMPLE_WALLS]
    cx, cy = inner_site
    polys.append([[cx - 0.12, cy - 0.1], [cx + 0.12, cy - 0.1], [cx, cy + 0.12]])
    walls = scenarios.pack_walls(polys)
    if per_env_shift is None:
        return walls
    walls = walls[None] + per_env_shift[:, None, None, None, :]
    for e in range(walls.shape[0]):  # keep endpoint order lexicographic after the shift (obstacle.py:31-32)
        for w in range(walls.shape[1]):
            for s in range(walls.shape[2]):
                if not np.isnan(walls[e, w, s, 0, 0]):
                    a, b = sorted([list(walls[e, w, s, 0]), list(walls[e, w, s, 1])])
                    walls[e, w, s, 0], walls[e, w, s, 1] = a, b
    return walls


def _scene(N, E, seed, spread=1.6, n_goals=None):
    """Crowd of _random_crowd, a visible holonomic robot at the clearest interior cell, walls at the edge and inside."""
    S, G = _random_crowd(E, N, seed, spread)
    sites, clear = _clear_cells(S, spread, 2)
    assert clear[0] > 0.38 and clear[1] > 0.3, clear   # room for the robot (0.3 m) and the inner obstacle without contact
    rob = np.zeros((E, 13))
    rob[:, 0:2] = sites[0]; rob[:, 8] = 0.3; rob[:, 9] = 80.0; rob[:, 12] = 1.0
    rob[:, 10:12] = sites[0] + [4.0, 3.0]
    act = np.random.RandomState(seed + 7).uniform(-0.4, 0.4, (E, 2))
    rob[:, 3:5] = act
    if n_goals is not None:
        G = _goal_lists(S, G, n_goals, seed)
    return S, G, rob, act, sites


def _goal_lists(S, G, n_goals, seed):
    """Goal lists of n_goals entries; a third of the humans start within their radius of goal 0 (switch at the first sub-step), a
    third are heading for a goal 0 they reach within the run, and the goal after it is near as well (a second switch)."""
    E, N = S.shape[:2]
    rng = np.random.RandomState(seed + 11)
    out = np.zeros((E, N, n_goals, 2))
    out[:, :, :] = rng.uniform(-2, 12, (E, N, n_goals, 2))
    out[:, :, :min(3, n_goals)] = G[:, :, :min(3, n_goals)]
    out[:, :, 2:][np.isnan(out[:, :, 2:])] = rng.uniform(-2, 12, int(np.isnan(out[:, :, 2:]).sum()))
    p, v, r = S[:, :, 0:2], S[:, :, 3:5], S[:, :, 8:9]
    u = v / np.maximum(np.linalg.norm(v, axis=-1, keepdims=True), 1e-9)
    sel = rng.randint(0, 3, (E, N))
    now = sel == 0
    out[now, 0] = p[now] + 0.5 * r[now] * u[now]
    soon = sel == 1
    out[soon, 0] = p[soon] + (r[soon] + 0.06) * u[soon]
    out[sel != 2, 1] = out[sel != 2, 0] + 0.3 * r[sel != 2] * u[sel != 2]
    return out


def _oracle_run(cfg, S1, G, walls, params, n, act, desired=None):
    E, N = G.shape[:2]
    D = np.zeros((E, N, 2)) if desired is None else desired
    return oracle.update_humans(cfg, S1, G, walls, params, np.zeros(S1.shape[:2]), D, DT, n, robot_vel=act, n_threads=THREADS)


def _assert_conditioned(cfg, S1, G, walls, params, act, ref):
    """The crowd, not the kernel: one-ulp perturbations of the positions must not move the oracle's own result by 1e-11."""
    rng = np.random.RandomState(0)
    Sp = S1.copy()
    N = G.shape[1]
    Sp[:, :N, 0:2] *= 1.0 + 2e-16 * rng.choice([-1.0, 1.0], Sp[:, :N, 0:2].shape)
    refp, _, _ = _oracle_run(cfg, Sp, G, walls, params, K, act)
    cond = _state_err(refp[:, :N], ref[:, :N])
    assert cond < 1e-11, f"ill-conditioned crowd ({cond:.2e}): use a larger spread"
    return cond


def _check_flags(eng, start, N, robot_start, act, time0, exact_touch):
    """Pre-step flags on the start state and post-step flags on the kernel's own end state, bit for bit against oracle.checks."""
    consts = np.array(eng.consts)
    r = eng.decode_flags()
    pre = oracle.checks(start, N, robot_start, act, time0, consts)
    assert np.array_equal(r["collision"], pre[:, 0] != 0) and np.array_equal(r["dmin"], pre[:, 1])
    assert np.array_equal(r["reaching_goal"], pre[:, 2] != 0) and np.array_equal(r["reward"], pre[:, 3])
    assert np.array_equal(r["terminated"], pre[:, 4] != 0) and np.array_equal(r["truncated"], pre[:, 5] != 0)
    assert np.array_equal(r["info"], pre[:, 6].astype(int))
    end = eng.rows(start)
    rob_end = eng.robot_rows()[0]
    post = oracle.checks(end, N, rob_end, act, time0, consts)
    assert np.array_equal(r["actual_collision"], post[:, 7] != 0) and np.array_equal(r["actual_dmin"], post[:, 8])
    assert np.array_equal(r["actual_goal"], post[:, 9] != 0)
    if exact_touch:   # one sub-step: touched during the run == overlapping at its end
        assert np.array_equal(r["touched"], post[:, 10] != 0)
    else:             # touched at any sub-step is implied by an overlap at the end
        assert np.all(r["touched"][post[:, 10] != 0])
    return pre, post


def _parity(model, N, dtype, seed, *, per_agent=False, per_env_walls=False, numba=False, symmetric=True, n_goals=None, section="state"):
    """The gym step (pre-checks, K sub-steps with the robot, post-checks, touch) against the oracle.  fp64: K sub-steps at 1e-9;
    fp32: one sub-step at 1e-4 from rounded inputs, then K sub-steps: finite, flags bit for bit."""
    from social_navigation_pyenvs_b200 import CrowdEngine
    E = _envs(N)
    S, G, rob, act, sites = _scene(N, E, seed, n_goals=n_goals)
    shift = np.random.RandomState(seed + 3).uniform(-0.2, 0.2, (E, 2)) if per_env_walls else None
    walls = _walls(S, 1.6, sites[1], shift)
    params = np.tile(oracle.default_params(model), (E, N, 1))
    if per_agent:
        rng = np.random.RandomState(seed + 5)
        params[:, :, 1] *= rng.uniform(0.8, 1.2, (E, N)); params[:, :, 3] *= rng.uniform(0.9, 1.1, (E, N))
        params[:, :, 0] *= rng.uniform(0.8, 1.2, (E, N))
    S1 = np.concatenate([S, rob[:, None]], 1)
    if dtype == torch.float32:
        S1, G, walls, act = _f32(S1, G, walls, act)
    sym = symmetric and not per_agent
    cfg = OracleConfig(oracle.type_code(model), True, sym, numba)

    def engine():
        eng = CrowdEngine.from_reference_arrays(model, S1, G, walls=walls, params=params if per_agent else None, consider_robot=True,
                                                all_params_equal=sym, numba_compat=numba, dtype=dtype)
        assert (eng.agent_params is not None) == per_agent and eng.walls_per_env == int(per_env_walls)
        return eng

    k = K if dtype == torch.float64 else 1
    eng = engine()
    eng.step(act, DT, n_substeps=k, pre_checks=True, post_checks=True, track_touch=True)
    got = eng.rows(S1)
    ref, Gr, Dr = _oracle_run(cfg, S1, G, walls, params, k, act)
    err = _state_err(got[:, :N], ref[:, :N])
    errf = float(rel_err(eng.desired_force(), Dr, scale=100.0).max())
    tol = 1e-9 if dtype == torch.float64 else 1e-4
    if dtype == torch.float64:
        _assert_conditioned(cfg, S1, G, walls, params, act, ref)
    _record(section, dtype, max(err, errf))
    assert err < tol and errf < tol, (err, errf)
    assert np.array_equal(got[:, :N, 10:12], ref[:, :N, 10:12])   # current goals (fp32: the same rounded goal)
    _check_flags(eng, S1, N, rob if dtype == torch.float64 else S1[:, N], act, np.zeros(E), exact_touch=k == 1)
    if dtype == torch.float32:
        eng = engine()
        eng.step(act, DT, n_substeps=K, pre_checks=True, post_checks=True, track_touch=True)
        assert np.isfinite(eng.rows(S1)).all() and np.isfinite(eng.desired_force()).all()
        _check_flags(eng, S1, N, S1[:, N], act, np.zeros(E), exact_touch=False)
    return ref, Gr


# ---------------------------------------------------------------------------------------------------------------------------
# 1. state parity across the mapping

def _model_cases():
    for N in SHAPES:
        models = MODELS if N in (65, 129, 512) else ["sfm_helbing", "hsfm_new_guo", "hsfm_moussaid"]
        for m in models:
            yield pytest.param(N, m, id=f"N{N}-{m}")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("N,model", list(_model_cases()))
def test_gym_step_vs_oracle(N, model, dtype):
    """Visible robot inside the crowd, walls at its edge and inside it, pre / post checks and touch on."""
    _parity(model, N, dtype, seed=N * 31 + MODELS.index(model))


VARIANTS = {
    "per_agent_params": dict(model="hsfm_guo", per_agent=True),          # the PER_AGENT instantiation (ordered loop)
    "per_env_walls": dict(model="sfm_guo", per_env_walls=True),          # wall staging per group, clamped in the ragged last CTA
    "numba_compat": dict(model="hsfm_new", numba=True),
    "moussaid_asymmetric": dict(model="sfm_moussaid", symmetric=False),  # sign(theta) of agent i, the ordered loop
    "goals4_cached": dict(model="hsfm_farina", n_goals=4),               # goal list staged in shared memory
    "goals5_global": dict(model="hsfm_farina", n_goals=5),               # goal list read from global memory
}


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("N", [43, 129])
def test_gym_step_variants_vs_oracle(N, variant, dtype):
    kw = dict(VARIANTS[variant])
    ref, Gr = _parity(kw.pop("model"), N, dtype, seed=N * 7 + list(VARIANTS).index(variant), section="variants", **kw)
    if "n_goals" in kw and dtype == torch.float64:   # the goal switches the case is about did happen within the run
        _, G, _, _, _ = _scene(N, _envs(N), N * 7 + list(VARIANTS).index(variant), n_goals=kw["n_goals"])
        moved = (ref[:, :N, 10:12] != G[:, :, 0]).any(-1)
        twice = (ref[:, :N, 10:12] == G[:, :, 2]).all(-1)
        assert moved.sum() >= N // 4 and twice.any(), (int(moved.sum()), int(twice.sum()))


# ---------------------------------------------------------------------------------------------------------------------------
# 2. checks, bit for bit

def _checks_scene(N, dtype, seed):
    """Robot away from the crowd, with a few humans moved next to it (their velocity = the action: the swept distance is the gap):
    env roles cover the five info codes, the first colliding human at 0, N/2, N-1 and beyond 128, a non-colliding human with a
    smaller swept distance right after it (a leader loop without the early break reports another dmin), and human 0 or N-1 as the
    human nearest to the robot (an admin loop that skips an end of the group reports another actual dmin)."""
    deep = 128 + (N - 128) // 2 if N > 128 else N // 3
    roles = [("collide", 0), ("collide", N // 2), ("collide", N - 1), ("collide", deep), ("danger", 0), ("danger", N - 1),
             ("goal", 0), ("goal", N - 1), ("timeout", N - 1), ("nothing", 0), ("nothing", N - 1)]
    E = len(roles)
    assert E % _gpb(N) != 0 or _gpb(N) == 1
    S, G = _random_crowd(E, N, seed, 1.6)
    rng = np.random.RandomState(seed + 1)
    act = rng.uniform(-0.4, 0.4, (E, 2))
    rob = np.zeros((E, 13))
    P = np.array([-3.5, -3.5])
    rob[:, 0:2] = P; rob[:, 3:5] = act; rob[:, 8] = 0.3; rob[:, 9] = 80.0; rob[:, 12] = 1.0; rob[:, 10:12] = P + [-6.0, 2.0]
    time0 = np.zeros(E)

    def put(e, i, gap, ang):
        S[e, i, 0:2] = P + (rob[e, 8] + S[e, i, 8] + gap) * np.array([np.cos(ang), np.sin(ang)])
        S[e, i, 3:5] = act[e]                      # zero velocity relative to the robot
    for e, (role, i) in enumerate(roles):
        if role == "collide":
            put(e, i, -0.05, 0.3)
            if i + 1 < N:
                put(e, i + 1, 0.01, 0.3 + np.pi)     # after the first collision, closer than anyone before it
            if i > 0:
                put(e, i - 1, 0.12, 0.3 + np.pi / 2)  # before it: the dmin the reference reports
        elif role == "danger":
            put(e, i, 0.1, 1.0)
            put(e, N // 2, 0.17, 1.0 + np.pi)
        elif role == "goal":
            rob[e, 10:12] = P + act[e] * 0.25       # the robot's end position: reaching_goal
            put(e, i, 0.3, 2.0)
        elif role == "timeout":
            time0[e] = 49.5
            put(e, i, 0.15, 2.5)
        else:
            put(e, i, 0.5, 0.5)
    S1 = np.concatenate([S, rob[:, None]], 1)
    if dtype == torch.float32:
        S1, G, act = _f32(S1, G, act)
        rob = S1[:, N].copy()
    return S1, G, rob, act, time0, roles


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("N", SHAPES)
def test_checks_bit_exact(N, dtype):
    """Pre-step and post-step reductions and the touch flag through shared memory, in the fused step (one sub-step) and through
    snp_checks (n_substeps = 0: both checks on the start state), and the swept test under the reference's own name."""
    from social_navigation_pyenvs_b200 import CrowdEngine
    S1, G, rob, act, time0, roles = _checks_scene(N, dtype, seed=N + 101)

    def engine():
        eng = CrowdEngine.from_reference_arrays("hsfm_farina", S1, G, consider_robot=True, all_params_equal=True, dtype=dtype)
        eng.time_now.copy_(torch.as_tensor(time0))
        return eng
    eng = engine()
    eng.step(act, DT, n_substeps=1, pre_checks=True, post_checks=True, track_touch=True)
    pre, post = _check_flags(eng, S1, N, rob, act, time0, exact_touch=True)
    assert set(pre[:, 6].astype(int)) == {0, 1, 2, 3, 4}
    assert pre[:, 0].sum() == 4 and post[:, 7].sum() >= 4 and post[:, 9].sum() >= 2 and post[:, 10].sum() >= 4
    # the nearest human at the end is the placed one (index 0 or N-1, or the first colliding one)
    end = eng.rows(S1)
    rob_end = eng.robot_rows()[0]
    d = np.linalg.norm(end[:, :N, 0:2] - rob_end[:, None, 0:2], axis=-1) - end[:, :N, 8] - rob_end[:, 8:9]
    assert [int(np.argmin(d[e])) for e in range(len(roles))] == [i for _, i in roles]
    # snp_checks: both checks on the start state
    eng = engine()
    r = eng.run_checks(act, pre=True, post=True)
    for key, col in (("dmin", 1), ("reward", 3), ("actual_dmin", 8)):
        assert np.array_equal(r[key], pre[:, col]), key
    for key, col in (("collision", 0), ("reaching_goal", 2), ("terminated", 4), ("truncated", 5), ("actual_collision", 7), ("actual_goal", 9)):
        assert np.array_equal(r[key], pre[:, col] != 0), key
    assert np.array_equal(r["info"], pre[:, 6].astype(int))
    col, dmin, goal = eng.collision_detection_and_reaching_goal(act, 0.25)
    assert np.array_equal(col, pre[:, 0] != 0) and np.array_equal(dmin, pre[:, 1]) and np.array_equal(goal, pre[:, 2] != 0)
    _record("checks", dtype, 0.0)


# ---------------------------------------------------------------------------------------------------------------------------
# 3. robot modes

def _robot_scene(N, E, seed):
    """Robot just left of the crowd with human 0 (even envs) or human N-1 (odd envs) nearest to it, 0.3 m from contact; in every
    other env the robot starts on its first goal (a goal switch at the first sub-step)."""
    S, G = _random_crowd(E, N, seed, 1.6)
    sites, _ = _clear_cells(S, 1.6, 1)
    rob = np.zeros((E, 13))
    P = np.array([-2.2, 0.5 * (S[:, :, 1].min() + S[:, :, 1].max())])
    rob[:, 0:2] = P; rob[:, 2] = 0.4; rob[:, 5:7] = [0.3, 0.1]; rob[:, 8] = 0.3; rob[:, 9] = 80.0; rob[:, 12] = 1.0
    c, s = np.cos(rob[:, 2]), np.sin(rob[:, 2])
    rob[:, 3], rob[:, 4] = c * rob[:, 5] - s * rob[:, 6], s * rob[:, 5] + c * rob[:, 6]
    rgoals = np.zeros((E, 2, 2))
    rgoals[:, 0] = P + [6.0, 1.0]
    rgoals[:, 1] = P + [-3.0, 4.0]
    rgoals[::2, 0] = P + [0.1, 0.05]
    for e in range(E):
        i = 0 if e % 2 == 0 else N - 1
        S[e, i, 0:2] = P + [0.0, rob[e, 8] + S[e, i, 8] + 0.3]
    rob[:, 10:12] = rgoals[:, 0]
    walls = _walls(S, 1.6, sites[0])
    return S, G, rob, rgoals, walls


def _robot_err(got_r, rr):
    cols = [0, 1, 3, 4, 5, 6, 7]
    e = float(rel_err(got_r[:, cols], rr[:, cols]).max())
    dth = (got_r[:, 2] - rr[:, 2] + np.pi) % (2 * np.pi) - np.pi
    return max(e, float((np.abs(dth) / np.maximum(np.abs(rr[:, 2]), 1.0)).max()))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("visible", [False, True], ids=["invisible", "visible"])
@pytest.mark.parametrize("N", [43, 129, 512])
def test_imitation_learning_step_vs_oracle(N, visible, dtype):
    """robot_mode 2, post_checks = 2: the robot moved by its own model (hsfm_new_guo, the humans' is hsfm_farina), its force summed
    over the group through shared memory, the actual checks and reward at the end."""
    from social_navigation_pyenvs_b200 import CrowdEngine
    E = _envs(N) + 2
    S, G, rob, rgoals, walls = _robot_scene(N, E, seed=N + 7)
    S1 = np.concatenate([S, rob[:, None]], 1) if visible else S
    if dtype == torch.float32:
        S1, G, rob, rgoals, walls = _f32(S1, G, rob, rgoals, walls)
    k = K if dtype == torch.float64 else 1
    eng = CrowdEngine.from_reference_arrays("hsfm_farina", S1, G, walls=walls, consider_robot=visible, all_params_equal=True, dtype=dtype,
                                            robot=None if visible else rob)
    eng.set_robot_motion_model("hsfm_new_guo", goals=rgoals)
    eng.imitation_learning_step(DT, n_substeps=k)
    cfg = OracleConfig(oracle.type_code("hsfm_farina"), visible, True, False)
    params = np.tile(oracle.default_params("hsfm_farina"), (E, N, 1))
    args = (cfg, S1, G, walls, params, np.zeros(S1.shape[:2]), np.zeros((E, N, 2)), DT)
    tail = (rob, rgoals, np.zeros((E, 2)), oracle.default_params("hsfm_new_guo"), oracle.type_code("hsfm_new_guo"))
    rh, rg, _, rr, _, _ = oracle.imitation_steps(*args, k, *tail, n_threads=THREADS)
    if dtype == torch.float64:
        Sp = S1.copy()
        Sp[:, :N, 0:2] *= 1.0 + 2e-16 * np.random.RandomState(0).choice([-1.0, 1.0], (E, N, 2))
        rhp, _, _, rrp, _, _ = oracle.imitation_steps(cfg, Sp, *args[2:], k, *tail, n_threads=THREADS)
        assert _state_err(rhp[:, :N], rh[:, :N]) < 1e-11 and _robot_err(rrp, rr) < 1e-11
    got = eng.rows(S1)
    got_r, _ = eng.robot_rows()
    err, errr = _state_err(got[:, :N], rh[:, :N]), _robot_err(got_r, rr)
    _record("robot", dtype, max(err, errr))
    tol = 1e-9 if dtype == torch.float64 else 1e-4
    assert err < tol and errr < tol, (err, errr)
    assert np.array_equal(got[:, :N, 10:12], rh[:, :N, 10:12])
    assert np.array_equal(got_r[:, 10:12], rr[:, 10:12]) and np.array_equal(got_r[::2, 10:12], rgoals[::2, 1])   # goal switch
    # actual checks and reward from the end state and end time (gym:269-271)
    f = eng.decode_flags()
    post = oracle.checks(got, N, got_r, np.zeros((E, 2)), eng.time_now.cpu().numpy(), np.array(eng.consts))   # the robot's current goal
    assert np.array_equal(f["actual_dmin"], post[:, 8]) and np.array_equal(f["actual_collision"], post[:, 7] != 0)
    assert np.array_equal(f["actual_goal"], post[:, 9] != 0)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("every", [1, 4])
@pytest.mark.parametrize("N", [43, 129, 512])
def test_sim_update_vs_oracle(N, every, dtype):
    """SocialNavSim.update with a model-driven visible robot: the humans see the robot's state from before its update; with
    robot_every = 4 the pose advances every update and the velocities are refreshed every fourth."""
    from social_navigation_pyenvs_b200 import CrowdEngine
    E = _envs(N)
    S, G, rob, rgoals, walls = _robot_scene(N, E, seed=N + 17)
    S1 = np.concatenate([S, rob[:, None]], 1)
    if dtype == torch.float32:
        S1, G, rob, rgoals, walls = _f32(S1, G, rob, rgoals, walls)
    k = K if dtype == torch.float64 else 1
    eng = CrowdEngine.from_reference_arrays("sfm_guo", S1, G, walls=walls, consider_robot=True, all_params_equal=True, dtype=dtype)
    eng.set_robot_motion_model("hsfm_farina", goals=rgoals)
    eng.sim_update(DT, n_updates=k, robot_every=every)
    cfg = OracleConfig(oracle.type_code("sfm_guo"), True, True, False)
    params = np.tile(oracle.default_params("sfm_guo"), (E, N, 1))
    rh, _, _, rr, _, _ = oracle.sim_update_steps(cfg, S1, G, walls, params, np.zeros((E, N + 1)), np.zeros((E, N, 2)), DT, k, rob, rgoals,
                                                 np.zeros((E, 2)), oracle.default_params("hsfm_farina"), oracle.type_code("hsfm_farina"),
                                                 every, DT * every, n_threads=THREADS)
    got = eng.rows(S1)
    got_r, _ = eng.robot_rows()
    err, errr = _state_err(got[:, :N], rh[:, :N]), _robot_err(got_r, rr)
    _record("robot", dtype, max(err, errr))
    tol = 1e-9 if dtype == torch.float64 else 1e-4
    assert err < tol and errr < tol, (err, errr)
    assert np.array_equal(got[:, :N, 10:12], rh[:, :N, 10:12])


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("N", [43, 129, 512])
def test_unicycle_robot_vs_oracle(N, dtype):
    """robot_mode 3 (ActionRot(v, r), robot_agent.py:116-136) with the robot inside the crowd: the oracle steps the humans once per
    sub-step around helpers.unicycle_step."""
    from social_navigation_pyenvs_b200 import CrowdEngine, _lib as L
    E = _envs(N)
    S, G, rob, _, sites = _scene(N, E, seed=N + 23)
    walls = _walls(S, 1.6, sites[1])
    rob[:, 2] = np.linspace(0.3, 2.8, E)
    rng = np.random.RandomState(N)
    action = np.stack([rng.uniform(0.3, 1.0, E), rng.uniform(-0.06, 0.06, E)], 1)
    S1 = np.concatenate([S, rob[:, None]], 1)
    if dtype == torch.float32:
        S1, G, walls, action = _f32(S1, G, walls, action)
    yaw = S1[:, N, 2].copy()
    k = K if dtype == torch.float64 else 1
    eng = CrowdEngine.from_reference_arrays("hsfm_new_guo", S1, G, walls=walls, consider_robot=True, all_params_equal=True, dtype=dtype)
    eng.robot[L.ROBOT_TH].copy_(torch.as_tensor(yaw, dtype=dtype))
    eng.step(action, DT, n_substeps=k, pre_checks=True, kinematics="unicycle")
    cfg = OracleConfig(oracle.type_code("hsfm_new_guo"), True, True, False)
    params = np.tile(oracle.default_params("hsfm_new_guo"), (E, N, 1))

    def run(S0):
        St, Gt, Dt, y = S0.copy(), G.copy(), np.zeros((E, N, 2)), yaw.copy()
        for _ in range(k):
            for e in range(E):
                St[e, N, 0:2], y[e], St[e, N, 3:5] = unicycle_step(St[e, N, 0:2], y[e], action[e, 0], action[e, 1], DT)
            St, Gt, Dt = oracle.update_humans(cfg, St, Gt, walls, params, np.zeros((E, N + 1)), Dt, DT, 1, n_threads=THREADS)
        return St, y
    ref, ryaw = run(S1)
    if dtype == torch.float64:
        Sp = S1.copy()
        Sp[:, :N, 0:2] *= 1.0 + 2e-16 * np.random.RandomState(0).choice([-1.0, 1.0], (E, N, 2))
        assert _state_err(run(Sp)[0][:, :N], ref[:, :N]) < 1e-11
    got = eng.rows(S1)
    err = _state_err(got[:, :N], ref[:, :N])
    _record("robot", dtype, err)
    assert err < (1e-9 if dtype == torch.float64 else 1e-4), err
    rb = eng.robot.double().cpu().numpy()
    rtol = 1e-12 if dtype == torch.float64 else 1e-5
    assert np.abs(rb[L.ROBOT_PX] - ref[:, N, 0]).max() < rtol and np.abs(rb[L.ROBOT_PY] - ref[:, N, 1]).max() < rtol
    assert np.abs(rb[L.ROBOT_TH] - ryaw).max() < rtol


# ---------------------------------------------------------------------------------------------------------------------------
# 4. peek and lookahead

@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("model", ["sfm_helbing", "hsfm_farina", "hsfm_new_moussaid"])
@pytest.mark.parametrize("N", [65, 129, 512])
def test_peek_vs_oracle(N, model, dtype):
    """get_next_human_observable_states and peek (dyn_out): one update into a side buffer; pose, velocities and goal index stay,
    the carried desired force is updated in place (mmm:691-709)."""
    from social_navigation_pyenvs_b200 import CrowdEngine, _lib as L
    E = _envs(N)
    S, G, rob, _, sites = _scene(N, E, seed=N + 41)
    S1 = np.concatenate([S, rob[:, None]], 1)
    D = np.random.RandomState(N).uniform(-50, 50, (E, N, 2))
    if dtype == torch.float32:
        S1, G, D = _f32(S1, G, D)
    dt = 0.25
    eng = CrowdEngine.from_reference_arrays(model, S1, G, consider_robot=True, all_params_equal=True, dtype=dtype)
    eng.set_desired_force(D)
    before, idx0 = eng.dyn[:8].clone(), eng.goal_idx.clone()
    obs = eng.get_next_human_observable_states(dt)
    cfg = OracleConfig(oracle.type_code(model), True, True, False)
    ref, _, Dr = oracle.update_humans(cfg, S1, G, None, np.tile(oracle.default_params(model), (E, N, 1)), np.zeros((E, N + 1)), D, dt, 1,
                                      n_threads=THREADS)
    tol = 1e-9 if dtype == torch.float64 else 1e-4
    err = float(rel_err(obs, ref[:, :N][..., [0, 1, 3, 4]]).max())
    errf = float(rel_err(eng.desired_force(), Dr, scale=100.0).max())
    _record("peek", dtype, max(err, errf))
    assert err < tol and errf < tol, (err, errf)
    assert torch.equal(eng.dyn[:8], before) and torch.equal(eng.goal_idx, idx0)
    # the raw side buffer: every field of the update
    eng.set_desired_force(D)
    nx = eng.peek(dt).double().cpu().numpy()
    cols = [(L.DYN_PX, 0), (L.DYN_PY, 1), (L.DYN_VX, 3), (L.DYN_VY, 4)] + ([(L.DYN_TH, 2), (L.DYN_BVX, 5), (L.DYN_BVY, 6), (L.DYN_OM, 7)]
                                                                          if eng.headed else [])
    for f, c in cols:
        g_c, r_c = nx[f], ref[:, :N, c]
        if f == L.DYN_TH:
            g_c = wrap_angle_cols(g_c[..., None], r_c[..., None], 0)[..., 0]
        assert rel_err(g_c, r_c).max() < tol, f
    assert torch.equal(eng.dyn[:8], before) and torch.equal(eng.goal_idx, idx0)


def _look_decomposition(N, E, A, visible, itemsize, sms):
    """launch_lookahead's choice (csrc/snp_lookahead.cu): (CTAs per env, actions per CTA, actions per tile, split by shared memory)."""
    OW = 15 if visible else 13
    per = max(256 // N, 1)
    while per > 1 and 2 * per * N * OW * itemsize > 64 * 1024:
        per -= 1
    splits = 1
    while splits < A and E * splits < 8 * 3 * sms:
        splits += 1
    by_sms = splits
    r16 = lambda x: (x + 15) & ~15
    pa_bytes = 16 + 8 * itemsize
    while True:
        aper = -(-A // splits)
        tiles = -(-aper // per)
        chunk = -(-aper // tiles)
        off = r16(itemsize * 11 * N)
        off = r16(off + pa_bytes * aper)
        off = r16(off + 8 * aper * N)
        total = off + 2 * r16(chunk * N * OW * itemsize + 16)
        if total <= 200 * 1024 or aper == 1:
            break
        splits += 1
    return -(-A // aper), aper, chunk, splits > by_sms


def _regime(N, E, A, visible, itemsize, sms):
    ctas, aper, chunk, by_smem = _look_decomposition(N, E, A, visible, itemsize, sms)
    if by_smem:
        return "smem_split"
    if aper == 1:
        return "aper1"
    if aper == A:
        return "whole_env"
    return "ragged" if A % aper else "even_split"


def _look_batch(E, N, seed):
    """Robots 3 m off the crowd's corner: near their goal (env 4k), 0.05 m from a human moved there at rest (4k+1: collisions
    and discomfort), 0.15 m from one (4k+2: discomfort), alone (4k+3)."""
    S, G = _random_crowd(E, N, seed, 1.1)
    rng = np.random.RandomState(seed)
    S[:, :, 3:5] = rng.uniform(-1, 1, (E, N, 2))
    R = np.zeros((E, 13))
    R[:, 0:2] = [-3.0, -3.0]
    R[:, 8], R[:, 9], R[:, 12] = 0.3, 80.0, 1.0
    R[:, 10:12] = R[:, 0:2] + [-4.0, -2.0]
    # a goal 0.5 m away, between two action directions: the fastest action towards it ends 0.26 m short of it (reached), and no
    # action ends so close to it that the rotation towards the goal (its direction from there) turns ill-conditioned in fp32
    R[::4, 10:12] = R[::4, 0:2] + 0.5 * np.array([np.cos(np.pi / 16), np.sin(np.pi / 16)])
    R[:, 2] = rng.uniform(-np.pi, np.pi, E)
    h = rng.randint(N, size=E)
    ang = rng.uniform(0, 2 * np.pi, E)
    for e in range(E):
        if e % 4 in (1, 2):
            gap = 0.05 if e % 4 == 1 else 0.15
            S[e, h[e], 0:2] = R[e, 0:2] + (0.3 + S[e, h[e], 8] + gap) * np.array([np.cos(ang[e]), np.sin(ang[e])])
            S[e, h[e], 3:5] = 0.0
    return S, G, R


def _lookahead_case(N, E, visible, dtype, model, sel=None):
    from social_navigation_pyenvs_b200 import CrowdEngine
    S, G, R = _look_batch(E, N, 5000 + N + E)
    acts = _actions()
    eng = CrowdEngine.from_reference_arrays(model, S, G, consider_robot=False, all_params_equal=True, robot=R, dtype=dtype)
    eng.set_action_space(acts)
    nxt = eng.peek(0.25)
    eng.lookahead_from(nxt, 0.25, theta_and_omega_visible=visible)   # allocates the outputs ...
    eng._rotated.fill_(float("nan")); eng._rewards.fill_(float("nan"))
    rot, rew = eng.lookahead_from(nxt, 0.25, theta_and_omega_visible=visible)   # ... which must be written word for word
    assert not torch.isnan(rot).any() and not torch.isnan(rew).any()
    sel = np.arange(E) if sel is None else sel
    cur, nxo, rob = _oracle_inputs(eng, nxt, visible, sel)
    rot_ref, rew_ref = oracle.lookahead(cur, nxo, rob, acts, 0.25, visible=visible, n_threads=THREADS)
    got_rew = rew.cpu().numpy()[sel]
    assert np.array_equal(got_rew, rew_ref)
    err = float(rel_err(rot[torch.as_tensor(sel, device=rot.device)].double().cpu().numpy(), rot_ref).max())
    _record("lookahead", dtype, err)
    assert err < (1e-9 if dtype == torch.float64 else 1e-4), err
    assert (rew_ref == -0.25).any() and (rew_ref == 1.0).any() and ((rew_ref < 0) & (rew_ref > -0.25)).any() and (rew_ref == 0).any()
    rot2, rew2 = rot.clone(), rew.clone()
    rot.zero_(); rew.zero_()
    rot3, rew3 = eng.lookahead_from(nxt, 0.25, theta_and_omega_visible=visible, bulk_store=False)
    assert torch.equal(rot2, rot3) and torch.equal(rew2, rew3)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("visible", [False, True], ids=["hidden", "visible"])
@pytest.mark.parametrize("N", [64, 129, 256, 257, 300, 512])
def test_lookahead_vs_oracle(N, visible, dtype):
    """E = 8: one action per CTA (aper = 1); N > 256 walks the tile with the strided loop (more pairs per tile than threads)."""
    assert _regime(N, 8, 81, visible, 8 if dtype == torch.float64 else 4, torch.cuda.get_device_properties(0).multi_processor_count) == "aper1"
    _lookahead_case(N, 8, visible, dtype, "hsfm_farina" if not visible else ("sfm_guo" if N % 2 else "hsfm_new_guo"))


# (N, E, visible, dtype, regime on a 148-SM B200): the decomposition of launch_lookahead each case reaches
REGIMES = [
    pytest.param(64, 1000, False, torch.float64, "ragged", id="ragged-N64-E1000-21.21.21.18-f64"),
    pytest.param(64, 1000, True, torch.float32, "ragged", id="ragged-N64-E1000-21.21.21.18-f32"),
    pytest.param(300, 200, True, torch.float64, "ragged", id="ragged-strided-N300-E200-5x16.1-f64"),
    pytest.param(300, 200, False, torch.float32, "ragged", id="ragged-strided-N300-E200-5x16.1-f32"),
    pytest.param(512, 400, True, torch.float64, "smem_split", id="smem_split-N512-E400-visible-f64"),
    pytest.param(64, 3600, False, torch.float64, "whole_env", id="whole_env-N64-E3600-f64"),
]


@pytest.mark.parametrize("N,E,visible,dtype,regime", REGIMES)
def test_lookahead_decomposition_regimes(N, E, visible, dtype, regime):
    """Ragged action split (the last CTA of each env takes fewer actions), a split forced by shared memory rather than by the SM
    count (about 2 GB of output), whole envs per CTA (1.9 GB); compared with the oracle on a sample of envs incl. the first and last."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert _regime(N, E, 81, visible, 8 if dtype == torch.float64 else 4, sms) == regime, sms
    sel = None if E <= 200 else np.r_[0:6, E // 2 - 3:E // 2 + 3, E - 6:E]
    _lookahead_case(N, E, visible, dtype, "hsfm_farina", sel)


def test_lookahead_decomposition_table():
    """The regimes named above, as launch_lookahead derives them for a 148-SM B200."""
    assert _look_decomposition(64, 1000, 81, False, 8, 148)[:2] == (4, 21)       # 21, 21, 21, 18
    assert _look_decomposition(300, 200, 81, True, 8, 148)[:2] == (17, 5)        # 16 x 5 + 1
    assert _look_decomposition(512, 400, 81, True, 8, 148)[3]
    assert _look_decomposition(64, 3600, 81, False, 8, 148)[:2] == (1, 81)
    assert _look_decomposition(512, 8, 81, False, 8, 148)[1] == 1


# ---------------------------------------------------------------------------------------------------------------------------
# 5. host-buffer step, respawn refusal

@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("N", [100, 512])
def test_step_host_equals_step(N, dtype):
    """snp_gym_step_host: the observation store of the block mapping into pinned buffers, and staged copies for pageable ones."""
    from social_navigation_pyenvs_b200 import CrowdEngine
    E = 5 if N == 100 else 3
    S, G, rob, _, sites = _scene(N, E, seed=N + 61)
    S1 = np.concatenate([S, rob[:, None]], 1)
    walls = _walls(S, 1.6, sites[1])
    mk = lambda: CrowdEngine.from_reference_arrays("hsfm_farina", S1, G, walls=walls, consider_robot=True, all_params_equal=True, dtype=dtype)
    a, b, d = mk(), mk(), mk()
    rng = np.random.RandomState(0)
    obs = torch.empty((4, E, N), dtype=dtype).pin_memory()
    flags = torch.empty((E,), dtype=torch.int32).pin_memory()
    checks = torch.empty((E, 4), dtype=torch.float64).pin_memory()
    obs3, flags3, checks3 = torch.empty((4, E, N), dtype=dtype), torch.empty((E,), dtype=torch.int32), torch.empty((E, 4), dtype=torch.float64)
    for _ in range(3):
        act = torch.as_tensor(rng.uniform(-0.4, 0.4, (2, E)), dtype=dtype).pin_memory()
        a.step_host(act, obs, flags, checks, DT, n_substeps=K, pre_checks=True, post_checks=True, track_touch=True)
        b.step(act.t().numpy(), DT, n_substeps=K, pre_checks=True, post_checks=True, track_touch=True)
        assert torch.equal(obs, b.dyn[:4].cpu()) and torch.equal(flags, b.flags.cpu()) and torch.equal(checks, b.checks.cpu())
        d.step_host(act.clone().numpy(), obs3, flags3, checks3, DT, n_substeps=K, pre_checks=True, post_checks=True, track_touch=True)
        assert torch.equal(obs3, obs) and torch.equal(flags3, flags) and torch.equal(checks3, checks)
    assert torch.equal(a.dyn, b.dyn) and torch.equal(a.robot, b.robot) and torch.equal(a.time_now, b.time_now)


def test_respawn_is_refused_above_32_humans():
    """Parallel-traffic respawn lives in the warp-packed mapping only: at N = 33 the step reports SNP_ERR_UNSUPPORTED
    (NotImplementedError) and changes nothing; N = 32 runs on the warp-packed mapping and matches the oracle."""
    from social_navigation_pyenvs_b200 import CrowdEngine
    for N in (33, 32):
        E = 5
        S, G = _random_crowd(E, N, N, 1.6)
        eng = CrowdEngine.from_reference_arrays("sfm_helbing", S, G, all_params_equal=True)
        eng.respawn_bounds = (7.0, 1.5)
        before = eng.dyn.clone()
        if N == 33:
            with pytest.raises(NotImplementedError):
                eng.update_humans(0.0, DT, n_substeps=1)
            torch.cuda.synchronize()
            assert torch.equal(eng.dyn, before)
        else:
            eng.update_humans(0.0, DT, n_substeps=1)
            cfg = OracleConfig(oracle.type_code("sfm_helbing"), False, True, False, (7.0, 1.5))
            ref, Gr, _ = oracle.update_humans(cfg, S, G, None, np.tile(oracle.default_params("sfm_helbing"), (E, N, 1)), np.zeros((E, N)),
                                              np.zeros((E, N, 2)), DT, 1)
            got = eng.rows(S)
            assert _state_err(got, ref) < 1e-9 and np.array_equal(got[..., 10:12], ref[..., 10:12])
