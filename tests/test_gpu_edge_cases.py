"""GPU parity at the degenerate ends of the shape range: a single human (no pair at all), two humans (only the antipodal
half-round of the halved pair loop), one env, the largest crowd of the fused kernel (512) and the first of the tiled one
(513), humans that start on their goal (the carried desired force of forces.py:9-16 and the goal rotation of mmm:66-70 with
one or two goals), and the error convention of the operator for empty inputs."""
import numpy as np
import pytest
import torch

import oracle
from oracle import OracleConfig
from helpers import rel_err
from test_gpu_sizes_large import _random_crowd

pytestmark = pytest.mark.gpu

WALL = [[[-2.0, -1.0], [-1.2, -1.0], [-1.2, 6.0], [-2.0, 6.0]]]


@pytest.mark.parametrize("robot", [False, True])
@pytest.mark.parametrize("model", ["hsfm_farina", "sfm_guo", "hsfm_new_moussaid"])
@pytest.mark.parametrize("N,E", [(1, 1), (1, 67), (2, 1), (2, 33), (4, 1), (6, 2), (512, 2)])
def test_degenerate_shapes_vs_oracle(model, N, E, robot):
    from social_navigation_pyenvs_b200 import CrowdEngine, scenarios
    S, G = _random_crowd(E, N, seed=7 * N + E, spread=1.1)
    rows, safety = S, np.full((E, N), 0.02)
    if robot:
        rob = np.zeros((E, 13)); rob[:, 0:2] = S[:, 0, 0:2] + 0.8; rob[:, 3:5] = [-0.3, 0.1]; rob[:, 8] = 0.3; rob[:, 9] = 80
        rows, safety = np.concatenate([S, rob[:, None]], 1), np.full((E, N + 1), 0.02)
    walls = scenarios.pack_walls(WALL)
    params = np.tile(oracle.default_params(model), (E, N, 1))
    cfg = OracleConfig(oracle.type_code(model), robot, True, False)
    ref, Gr, Dr = oracle.update_humans(cfg, rows, G, walls, params, safety, np.zeros((E, N, 2)), 0.0125, 3, n_threads=4)
    eng = CrowdEngine.from_reference_arrays(model, rows, G, walls=walls, safety=safety, consider_robot=robot, all_params_equal=True)
    eng.update_humans(0.0, 0.0125, n_substeps=3)
    got = eng.rows(rows)
    assert np.isfinite(got[:, :N, :8]).all()
    tol = 1e-9 if "moussaid" not in model else 1e-6   # moving crowd: no at-rest sign ambiguity, but atan2 differs in the last ulps
    assert rel_err(got[:, :N, :8], ref[:, :N, :8]).max() < tol
    assert np.array_equal(got[:, :N, 10:12], ref[:, :N, 10:12])
    assert rel_err(eng.desired_force(), Dr, scale=100.0).max() < 1e-9


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-9), (torch.float32, 1e-4)])
def test_first_crowd_of_the_tiled_kernel_vs_oracle(dtype, tol):
    """513 humans: one more than the fused kernel takes (snp_step answers SNP_ERR_UNSUPPORTED -> NotImplementedError and names
    snp_large_run_p2p); the tiled all-pairs kernels take it, with a ragged last tile."""
    from social_navigation_pyenvs_b200 import CrowdEngine
    from social_navigation_pyenvs_b200.large import LargeCrowd
    n = 513
    S, G = _random_crowd(1, n, seed=513, spread=1.1)
    if dtype == torch.float64:
        with pytest.raises(NotImplementedError, match="snp_large_run_p2p"):
            CrowdEngine.from_reference_arrays("hsfm_farina", S, G, all_params_equal=True).update_humans(0.0, 0.0125)
    if dtype == torch.float32:
        S = S.astype(np.float32).astype(np.float64); G = G.astype(np.float32).astype(np.float64)
    cfg = OracleConfig(oracle.type_code("hsfm_farina"), False, True, False)
    params = np.tile(oracle.default_params("hsfm_farina"), (1, n, 1))
    ref, _, _ = oracle.update_humans(cfg, S, G, None, params, np.zeros((1, n)), np.zeros((1, n, 2)), 0.0125, 1)
    crowd = LargeCrowd("hsfm_farina", S[0], G[0], dtype=dtype, symmetric=True)
    crowd.step(0.0125, n_substeps=1)
    assert rel_err(crowd.local_rows(S[0])[:, :8], ref[0, :, :8]).max() < tol


@pytest.mark.parametrize("n_goals", [1, 2])
@pytest.mark.parametrize("model", ["sfm_helbing", "hsfm_farina"])
def test_humans_starting_on_their_goal(model, n_goals):
    """Inside the goal radius the desired force is NOT recomputed (forces.py:12 `if dist > radius`): the carried value is used,
    and the goal list rotates first (mmm:66-70) -- onto itself when it holds a single goal."""
    from social_navigation_pyenvs_b200 import CrowdEngine
    E, N = 9, 5
    S, G3 = _random_crowd(E, N, seed=11, spread=1.5)
    G = np.full((E, N, 2, 2), np.nan)
    G[:, :, 0] = S[:, :, 0:2] + 0.05                   # inside every radius (>= 0.25)
    G[:, 0::2, 0] = S[:, 0::2, 0:2]                   # and exactly ON the goal for every other human (distance 0)
    if n_goals == 2:
        G[:, :, 1] = G3[:, :, 1]
    S[:, :, 10:12] = G[:, :, 0]
    D0 = np.random.RandomState(2).uniform(-30, 30, (E, N, 2))   # the carried desired force of the previous step
    params = np.tile(oracle.default_params(model), (E, N, 1))
    cfg = OracleConfig(oracle.type_code(model), False, True, False)
    ref, Gr, Dr = oracle.update_humans(cfg, S, G, None, params, np.zeros((E, N)), D0, 0.0125, 2, n_threads=2)
    eng = CrowdEngine.from_reference_arrays(model, S, G, all_params_equal=True)
    eng.set_desired_force(D0)
    eng.update_humans(0.0, 0.0125, n_substeps=2)
    got = eng.rows(S)
    assert np.isfinite(got[:, :, :8]).all()
    assert rel_err(got[:, :, :8], ref[:, :, :8]).max() < 1e-9
    assert np.array_equal(got[:, :, 10:12], ref[:, :, 10:12])
    assert rel_err(eng.desired_force(), Dr, scale=100.0).max() < 1e-9


def test_operator_rejects_empty_crowds():
    """The reference has no notion of an empty crowd (the Numba operator indexes row 0); the C ABI answers SNP_ERR_INVALID and
    the host operator raises ValueError, as for a bad type (fp:211)."""
    from social_navigation_pyenvs_b200 import update_humans_parallel
    with pytest.raises(ValueError):
        update_humans_parallel(3, np.zeros((0, 13)), np.zeros((0, 1, 2)), None, np.zeros((0, 20)), 0.0125, np.zeros(0))
