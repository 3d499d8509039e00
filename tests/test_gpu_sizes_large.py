"""GPU parity at other crowd shapes: lane packing (N=5, several envs per warp, ragged last warp), CTA-per-env (N > 32),
per-env walls, per-agent parameter rows, the host operator with serial semantics, and the large tiled all-pairs kernel."""
import os

import numpy as np
import pytest
import torch

import oracle
from oracle import OracleConfig
from helpers import load_traj, rel_err, inputs_at, observed, traj_names

pytestmark = pytest.mark.gpu


def _random_crowd(E, N, seed, spread):
    rng = np.random.RandomState(seed)
    S = np.zeros((E, N, 13))
    # jittered grid so nobody overlaps too deeply but neighbours interact
    side = int(np.ceil(np.sqrt(N)))
    gx, gy = np.meshgrid(np.arange(side), np.arange(side), indexing="ij")
    base = np.stack([gx.ravel(), gy.ravel()], 1)[:N] * spread
    S[:, :, 0:2] = base[None] + rng.uniform(-0.3, 0.3, (E, N, 2)) * spread
    S[:, :, 2] = rng.uniform(-np.pi, np.pi, (E, N))
    S[:, :, 5:7] = rng.uniform(-0.5, 0.5, (E, N, 2))
    S[:, :, 7] = rng.uniform(-0.3, 0.3, (E, N))
    c, s = np.cos(S[:, :, 2]), np.sin(S[:, :, 2])
    S[:, :, 3] = c * S[:, :, 5] - s * S[:, :, 6]
    S[:, :, 4] = s * S[:, :, 5] + c * S[:, :, 6]
    S[:, :, 8] = rng.uniform(0.25, 0.45, (E, N))
    S[:, :, 9] = rng.uniform(60, 90, (E, N))
    S[:, :, 12] = rng.uniform(0.6, 1.4, (E, N))
    G = np.full((E, N, 3, 2), np.nan)
    G[:, :, 0] = rng.uniform(-2, side * spread + 2, (E, N, 2))
    G[:, :, 1] = rng.uniform(-2, side * spread + 2, (E, N, 2))
    some = rng.rand(E, N) < 0.5
    G[some, 2] = rng.uniform(-2, side * spread + 2, (int(some.sum()), 2))
    S[:, :, 10:12] = G[:, :, 0]
    return S, G


@pytest.mark.parametrize("model", ["sfm_helbing", "sfm_guo", "hsfm_farina", "hsfm_new_guo", "hsfm_moussaid"])
@pytest.mark.parametrize("N,E", [(5, 1001), (3, 77), (16, 130), (31, 40), (32, 9), (33, 6), (100, 5), (300, 3)])
def test_shapes_vs_oracle(model, N, E):
    """Every thread mapping of snp_step: warp-packed (several envs per warp, ragged tail), one env per warp, CTA per env."""
    from social_navigation_pyenvs_b200 import CrowdEngine
    S, G = _random_crowd(E, N, seed=N * 1000 + E, spread=1.1)
    rob = np.zeros((E, 13)); rob[:, 0:2] = S[:, 0, 0:2] + 0.9; rob[:, 3:5] = [0.3, -0.2]; rob[:, 8] = 0.3; rob[:, 9] = 80
    S1 = np.concatenate([S, rob[:, None]], 1)
    safety = np.full((E, N + 1), 0.03)
    params = np.tile(oracle.default_params(model), (E, N, 1))
    cfg = OracleConfig(oracle.type_code(model), True, True, False)
    k = 3
    ref, Gr, Dr = oracle.update_humans(cfg, S1, G, None, params, safety, np.zeros((E, N, 2)), 0.0125, k, n_threads=4)
    eng = CrowdEngine.from_reference_arrays(model, S1, G, safety=safety, consider_robot=True, all_params_equal=True)
    eng.update_humans(0.0, 0.0125, n_substeps=k)
    got = eng.rows(S1)
    assert rel_err(got[:, :N, :8], ref[:, :N, :8]).max() < 1e-9
    assert np.array_equal(got[:, :N, 10:12], ref[:, :N, 10:12])
    assert rel_err(eng.desired_force(), Dr, scale=100.0).max() < 1e-9


@pytest.mark.parametrize("N,E", [(5, 203), (25, 37), (12, 50), (32, 11)])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_warp_packed_and_block_packed_mappings_agree(N, E, dtype):
    """The same crowd through both thread mappings (envs tiling warps vs envs tiling a 128-thread CTA), with walls, robot, checks
    and 10 fused sub-steps: states within rounding of each other and of the oracle, flags identical."""
    from social_navigation_pyenvs_b200 import CrowdEngine, scenarios
    S, G = _random_crowd(E, N, seed=N + E, spread=2.0)  # roomy crowd: 10 fused sub-steps must not amplify rounding chaotically
    rob = np.zeros((E, 13)); rob[:, 0:2] = [-1.7, -1.7];  # clear of every human: a deep overlap makes the dynamics chaotic
    rob[:, 3:5] = [0.2, -0.1]; rob[:, 8] = 0.3; rob[:, 9] = 80; rob[:, 10:12] = 5.0
    S1 = np.concatenate([S, rob[:, None]], 1)
    if dtype == torch.float32:
        S1 = S1.astype(np.float32).astype(np.float64); G = G.astype(np.float32).astype(np.float64)
    walls = scenarios.pack_walls([[[-2.0, -1.0], [-1.2, -1.0], [-1.2, 6.0], [-2.0, 6.0]]])
    act = np.tile([0.2, -0.1], (E, 1))
    out = []
    for mapping in (1, 2):
        eng = CrowdEngine.from_reference_arrays("hsfm_new_guo", S1, G, walls=walls, consider_robot=True, all_params_equal=True, dtype=dtype)
        eng.mapping = mapping
        eng.step(act, 0.0125, n_substeps=10, pre_checks=True, post_checks=True, track_touch=True)
        out.append((eng.rows(S1), eng.flags.cpu().numpy().copy(), eng.checks.cpu().numpy().copy(), eng.robot.cpu().numpy().copy()))
    tol = 1e-10 if dtype == torch.float64 else 2e-3
    assert rel_err(out[0][0][:, :N, :8], out[1][0][:, :N, :8]).max() < tol
    assert np.array_equal(out[0][1] & 0x7F, out[1][1] & 0x7F) and np.array_equal(out[0][2][:, :2], out[1][2][:, :2])   # pre-step flags / dmin / reward
    assert np.array_equal(out[0][3], out[1][3])
    if dtype == torch.float64:
        cfg = OracleConfig(oracle.type_code("hsfm_new_guo"), True, True, False)
        params = np.tile(oracle.default_params("hsfm_new_guo"), (E, N, 1))
        ref, _, _ = oracle.update_humans(cfg, S1, G, walls, params, np.zeros((E, N + 1)), np.zeros((E, N, 2)), 0.0125, 10, robot_vel=act, n_threads=4)
        assert rel_err(out[1][0][:, :N, :8], ref[:, :N, :8]).max() < 1e-9


def test_per_env_walls_and_per_agent_params():
    from social_navigation_pyenvs_b200 import CrowdEngine, scenarios
    E, N = 37, 7
    S, G = _random_crowd(E, N, seed=5, spread=1.3)
    rng = np.random.RandomState(3)
    base = scenarios.pack_walls([[[-1.5, -1.0], [-1.0, -1.0], [-1.0, 4.0], [-1.5, 4.0]], [[0.5, 4.6], [3.0, 4.6], [1.7, 5.5]]])
    walls = base[None] + rng.uniform(-0.2, 0.2, (E, 1, 1, 1, 2))
    for e in range(E):  # keep endpoint order lexicographic after the shift (obstacle.py:31-32)
        for w in range(walls.shape[1]):
            for s in range(walls.shape[2]):
                if not np.isnan(walls[e, w, s, 0, 0]):
                    a, b = sorted([list(walls[e, w, s, 0]), list(walls[e, w, s, 1])])
                    walls[e, w, s, 0], walls[e, w, s, 1] = a, b
    params = np.tile(oracle.default_params("hsfm_guo"), (E, N, 1))
    params[:, :, 1] *= rng.uniform(0.8, 1.2, (E, N)); params[:, :, 17] *= rng.uniform(0.8, 1.2, (E, N))
    cfg = OracleConfig(oracle.type_code("hsfm_guo"), False, False, False)
    ref, _, Dr = oracle.update_humans(cfg, S, G, walls, params, np.zeros((E, N)), np.zeros((E, N, 2)), 0.0125, 2)
    eng = CrowdEngine.from_reference_arrays("hsfm_guo", S, G, walls=walls, params=params, all_params_equal=False)
    assert eng.agent_params is not None and eng.walls_per_env == 1
    eng.update_humans(0.0, 0.0125, n_substeps=2)
    assert rel_err(eng.rows(S)[:, :, :8], ref[:, :, :8]).max() < 1e-9


@pytest.mark.parametrize("name", ["walls7_hsfm_guo", "walls7eq_sfm_guo", "corridor_hsfm_new", "ccso8_hsfm_farina", "cc7_randattr_sfm_helbing"])
def test_host_operator_serial_semantics_with_carried_desired_force(name):
    """update_humans_parallel(...) drop-in with host arrays: default semantics = the serial Python/NumPy path; goals are rotated in
    place and the goal columns of the input are refreshed like the reference does (fp:229-234)."""
    from social_navigation_pyenvs_b200 import update_humans_parallel
    d = load_traj(name)
    n = d["n"]
    S, G, D, rv = inputs_at(d, 0)
    saf = d["safety"][: S.shape[0]]
    walls = d["walls"] if d["walls"].shape[0] else None
    cur = 0
    for k, s in enumerate(d["steps"][:12]):
        while cur < s:
            if d["consider_robot"]:
                S[n, 0:2] = S[n, 0:2] + rv * float(d["dt"]); S[n, 3:5] = rv
            out = update_humans_parallel(int(d["type"]), S, G, walls, d["params"], float(d["dt"]), saf, all_params_equal=d["all_equal"],
                                         last_is_robot=d["consider_robot"], desired_force=D)
            assert np.array_equal(S[:n, 10:12], out[:n, 10:12]) and np.array_equal(G[:, 0], out[:n, 10:12])
            S = out
            cur += 1
        got = observed(S, D, n)
        assert rel_err(got[:, :10], d["traj"][k][:, :10]).max() < 1e-9, (name, int(s))


def test_large_crowd_tiled_kernel_vs_oracle():
    """snp_large_run_p2p on a 1024-human crowd (type 3 and 7, walls) against the oracle's row-major pair loop, 3 sub-steps."""
    from social_navigation_pyenvs_b200 import scenarios
    from social_navigation_pyenvs_b200.large import LargeCrowd
    sc = scenarios.jittered_grid_crowd(32, pitch=1.0, jitter=0.3, seed=0)
    S, G = sc["states"], sc["goals"]
    n = S.shape[1]
    rng = np.random.RandomState(0)
    S[0, :, 5:7] = rng.uniform(-0.6, 0.6, (n, 2)); S[0, :, 7] = rng.uniform(-0.2, 0.2, n)
    c, s_ = np.cos(S[0, :, 2]), np.sin(S[0, :, 2])  # moving crowd (Moussaid from rest is ill-defined, see helpers.py)
    S[0, :, 3] = c * S[0, :, 5] - s_ * S[0, :, 6]; S[0, :, 4] = s_ * S[0, :, 5] + c * S[0, :, 6]
    walls = scenarios.pack_walls([[[-3.0, -20.0], [-2.5, -20.0], [-2.5, 20.0], [-3.0, 20.0]]])
    for model in ["hsfm_farina", "hsfm_new_guo", "sfm_moussaid"]:
        cfg = OracleConfig(oracle.type_code(model), False, True, False)
        params = np.tile(oracle.default_params(model), (1, n, 1))
        ref, _, Dr = oracle.update_humans(cfg, S, G, walls, params, np.zeros((1, n)), np.zeros((1, n, 2)), 0.0125, 3)
        crowd = LargeCrowd(model, S[0], G[0], walls=walls, symmetric=True)
        crowd.step(0.0125, n_substeps=3)
        got = crowd.local_rows(S[0])
        tol = 1e-9 if "moussaid" not in model else 1e-6
        assert rel_err(got[:, :8], ref[0, :, :8]).max() < tol, model


@pytest.mark.parametrize("order", ["row_major", "patch"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_large_crowd_chunked_sums_and_exact_culling(dtype, order):
    """5184 humans (41 j-chunks and tiles, a 72 m wide crowd): the chunked partial sums stay within 1e-9 of the oracle's single
    j-ascending sum, and skipping tiles beyond the exp-underflow distance changes NOTHING (bit-identical on/off) -- with the
    humans numbered row by row (long thin tiles) or patch by patch (scenarios.spatial_order: compact tiles, more of them culled);
    on the whole crowd (culled on the work list) and on a slice that does not start on a tile (culled on the static grid)."""
    from social_navigation_pyenvs_b200 import scenarios
    from social_navigation_pyenvs_b200.large import LargeCrowd
    sc = scenarios.jittered_grid_crowd(72, pitch=1.0, jitter=0.3, seed=3)
    S, G = sc["states"], sc["goals"]
    n = S.shape[1]
    if order == "patch":
        perm = scenarios.spatial_order(S[0, :, 0:2])
        assert np.array_equal(np.sort(perm), np.arange(n))
        S, G = np.ascontiguousarray(S[:, perm]), np.ascontiguousarray(G[:, perm])
    rng = np.random.RandomState(1)
    S[0, :, 5:7] = rng.uniform(-0.6, 0.6, (n, 2))
    if dtype == torch.float32:
        S = S.astype(np.float32).astype(np.float64)
    out = {}
    # the whole crowd: culled on the list of near (i-block, chunk) pairs worked off by persistent CTAs, or all pairs; a slice at
    # offset 64: culled on the static grid, or all pairs
    for shard in (None, (64, n - 64)):
        for cull in (True, False):
            crowd = LargeCrowd("hsfm_farina", S[0], G[0], dtype=dtype, symmetric=True, shard=shard)
            crowd.culling = cull
            rows = S[0] if shard is None else S[0, 64:]
            crowd.step(0.0125, n_substeps=2)
            first = crowd.local_rows(rows)
            crowd.step(0.0125, n_substeps=1)  # (a second call: the list's counters were left empty by the first)
            out[shard, cull] = (first, crowd.local_rows(rows))
        for k in (0, 1):
            assert np.array_equal(out[shard, True][k], out[shard, False][k]), (shard, k)
    out = {True: out[None, True][0]}
    cfg = OracleConfig(oracle.type_code("hsfm_farina"), False, True, False)
    params = np.tile(oracle.default_params("hsfm_farina"), (1, n, 1))
    ref, _, _ = oracle.update_humans(cfg, S, G, None, params, np.zeros((1, n)), np.zeros((1, n, 2)), 0.0125, 2)
    tol = 1e-9 if dtype == torch.float64 else 1e-4
    assert rel_err(out[True][:, :8], ref[0, :, :8]).max() < tol


@pytest.mark.parametrize("case", ["shard_substeps_in_one_call", "nccl_vs_fused"])
def test_large_crowd_same_bits_however_the_substeps_are_called(case):
    """fp32 hsfm_farina (culling reach 88 B ~ 7 m), sub-steps compared bit for bit:
    * a shard= slice (the first 1024 humans of a 72 x 72 crowd numbered row by row: x ~ -35 m, away from the crowd's centre) stepped
      3 sub-steps in one call == 3 calls of one: the tile boxes of the frozen rest of the crowd are recomputed every sub-step, not
      read from a next-view table its producers only partly wrote;
    * a 1024-human crowd with exchange="nccl" forced on one GPU (one C call per sub-step, then the all-gather) == the fused one
      (the sub-step loop in one C call, tile boxes written by the producers), over two calls of several sub-steps each."""
    from social_navigation_pyenvs_b200 import model_parameters, scenarios
    from social_navigation_pyenvs_b200.large import LargeCrowd
    side = 72 if case == "shard_substeps_in_one_call" else 32
    sc = scenarios.jittered_grid_crowd(side, pitch=1.0, jitter=0.3, seed=4)
    S, G = sc["states"][0], sc["goals"][0]
    S[:, 5:7] = np.random.RandomState(2).uniform(-0.6, 0.6, (S.shape[0], 2))
    if case == "shard_substeps_in_one_call":
        shard, rows = (0, 1024), S[:1024]
        reach = 88 * model_parameters("hsfm_farina")[3] + 2 * S[:, 8].max() + 0.1
        assert S[1024:, 0].min() - S[:1024, 0].max() < reach < S[:, 0].max() - S[:1024, 0].max()  # neighbours in reach, units culled
        assert S[:1024, 0].max() < -reach  # the zero boxes the next view's table starts with sit at the origin, out of reach
        a = LargeCrowd("hsfm_farina", S, G, dtype=torch.float32, symmetric=True, shard=shard)
        b = LargeCrowd("hsfm_farina", S, G, dtype=torch.float32, symmetric=True, shard=shard)
        assert a.exchange == b.exchange == "fused"
        a.step(0.0125, n_substeps=3)
        for _ in range(3):
            b.step(0.0125, n_substeps=1)
    else:
        rows = S
        a = LargeCrowd("hsfm_farina", S, G, dtype=torch.float32, symmetric=True)
        b = LargeCrowd("hsfm_farina", S, G, dtype=torch.float32, symmetric=True, exchange="nccl")
        assert (a.exchange, b.exchange) == ("fused", "nccl")
        for k in (3, 2):
            a.step(0.0125, n_substeps=k)
            b.step(0.0125, n_substeps=k)
    assert np.array_equal(a.local_rows(rows), b.local_rows(rows))


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("workload", ["4096x25_hsfm_ccso_walls_robot", "4096x5_sfm_helbing_cc"])
def test_state_parity_at_the_bench_configurations(workload, dtype):
    """BASELINE configs[2] and configs[1] at their FULL size (4096 envs), the crowds bench.py times: the state after one fused
    launch of 20 sub-steps against the oracle (fp64: 1e-9 relative; fp32: 1e-4 after ONE sub-step -- north_star's per-step bar --
    and the accumulated figure after 20 reported through a looser bound)."""
    import oracle
    from oracle import OracleConfig
    from social_navigation_pyenvs_b200 import CrowdEngine, scenarios
    model, E, N, with_walls, visible = {"4096x25_hsfm_ccso_walls_robot": ("hsfm_farina", 4096, 25, True, True),
                                        "4096x5_sfm_helbing_cc": ("sfm_helbing", 4096, 5, False, False)}[workload]
    sc = scenarios.ccso_synthetic(E, N, 2000) if with_walls else scenarios.circular_crossing(E, N, 2000)
    walls = scenarios.pack_walls(scenarios.EXAMPLE_WALLS) if with_walls else None
    states = np.concatenate([sc["states"], sc["robot"][:, None]], 1) if visible else sc["states"]
    safety = np.zeros(states.shape[:2])
    action = np.tile([0.0, 1.0], (E, 1))
    cfg = OracleConfig(oracle.type_code(model), visible, True, False)
    params = np.tile(oracle.default_params(model), (E, N, 1))
    for k, tol64, tol32 in ((1, 1e-9, 1e-4), (20, 1e-9, 2e-3)):
        eng = CrowdEngine.from_reference_arrays(model, states, sc["goals"], walls=walls, safety=safety, consider_robot=visible, all_params_equal=True,
                                                dtype=dtype, robot=None if visible else sc["robot"])
        eng.step(action, 0.0125, n_substeps=k, pre_checks=True, track_touch=True)
        got = eng.rows(states)
        ref, _, _ = oracle.update_humans(cfg, states, sc["goals"], walls, params, safety, np.zeros((E, N, 2)), 0.0125, k,
                                         robot_vel=action if visible else None, n_threads=os.cpu_count() or 1)
        g, r = got[:, :N, :8].copy(), ref[:, :N, :8]
        g[..., 2] = r[..., 2] + (g[..., 2] - r[..., 2] + np.pi) % (2 * np.pi) - np.pi   # headings compared as angles
        err = rel_err(g, r).max()
        assert err < (tol64 if dtype == torch.float64 else tol32), (workload, k, float(err))
        if dtype == torch.float64:
            assert np.array_equal(got[:, :N, 10:12], ref[:, :N, 10:12])   # current goals: exact
        else:                                                              # (the same goal, stored in single precision)
            assert np.abs(got[:, :N, 10:12] - ref[:, :N, 10:12]).max() < 1e-5
