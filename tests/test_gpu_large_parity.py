"""The large-crowd path (snp_large_run_p2p) against the oracle and against itself, with the scratch and the tile-box tables
poisoned before every call, so that a read of anything the same sub-step did not write shows up:

* every model in fp64 and fp32 on a moving ~1500-human crowd (ragged last tile) with per-human safety, the three example wall
  polygons inside the crowd and two-goal lists that some humans finish during the run;
* numba_compat semantics, symmetric=False, and a wall set whose staged segments need more than 48 KB of shared memory;
* slices (shard=) of the 72 x 72 crowd that start on or off a tile and fill or do not fill their last one: the same bits as the
  whole crowd's rows, as all pairs, and as one sub-step per call;
* the culling reach: a lone human just inside or just outside it."""
import functools

import numpy as np
import pytest
import torch

import oracle
from oracle import OracleConfig
from helpers import rel_err, wrap_angle_cols

pytestmark = pytest.mark.gpu

SFMS = oracle.SFMS
DT = 0.0125


def _poison(crowd, whole):
    """Before a step call: the scratch all ones (NaN as fp32 and fp64, -1 as int32); the tile boxes of both view buffers far away
    (a stale box then drops forces; a NaN box would only compare as near); for a whole-crowd run also the entries of the view the
    call writes.  A shard= run keeps them: the frozen rest of the crowd lives there."""
    crowd.scratch.fill_(0xFF)
    M = crowd.n_total
    for v in crowd._vbuf:
        boxes = v[5 * M:].view(crowd._n_tiles, 5)
        boxes[:, :4] = 1e30
        boxes[:, 4] = 0.0
    if whole:
        crowd._vbuf[crowd.cur ^ 1][:5 * M].fill_(float("nan"))


def _step(crowd, k, whole=True):
    _poison(crowd, whole)
    crowd.step(DT, n_substeps=k)


def _f32(*arrays):
    return [None if a is None else np.asarray(a, np.float64).astype(np.float32).astype(np.float64) for a in arrays]


def _moving(S, rng):
    """Random body velocities and angular velocities; the world-frame velocity from the heading (mmm:448)."""
    n = S.shape[0]
    S[:, 5:7] = rng.uniform(-0.6, 0.6, (n, 2))
    S[:, 7] = rng.uniform(-0.2, 0.2, n)
    c, s = np.cos(S[:, 2]), np.sin(S[:, 2])
    S[:, 3] = c * S[:, 5] - s * S[:, 6]
    S[:, 4] = s * S[:, 5] + c * S[:, 6]


def _crowd_with_walls(polygons, clearance, seed):
    """A moving 39 x 39 jittered grid without the humans near the wall polygons, with per-human safety and goals that some
    humans reach during the run: 40 start within the goal radius (switch on the first sub-step), 40 a few sub-steps of travel
    outside it along their velocity."""
    from social_navigation_pyenvs_b200 import scenarios
    sc = scenarios.jittered_grid_crowd(39, pitch=1.0, jitter=0.3, seed=seed)
    S, G = sc["states"][0], sc["goals"][0]
    keep = np.ones(len(S), bool)
    for poly in polygons:
        p = np.asarray(poly, np.float64)
        keep &= ~np.all((S[:, 0:2] > p.min(0) - clearance) & (S[:, 0:2] < p.max(0) + clearance), axis=1)
    S, G = np.ascontiguousarray(S[keep]), np.ascontiguousarray(G[keep])
    n = len(S)
    rng = np.random.RandomState(seed + 100)
    _moving(S, rng)
    safety = rng.uniform(0.0, 0.1, n)
    pick = rng.choice(n, 80, replace=False)
    inside, ahead = pick[:40], pick[40:]
    G[pick, 1] = G[pick, 0]  # the next goal: across the crowd
    ang = rng.uniform(-np.pi, np.pi, 40)
    dist = S[inside, 8] - rng.uniform(0.02, 0.05, 40)
    G[inside, 0] = S[inside, 0:2] + dist[:, None] * np.stack([np.cos(ang), np.sin(ang)], 1)
    v = S[ahead, 3:5]
    sp = np.linalg.norm(v, axis=1, keepdims=True)
    G[ahead, 0] = S[ahead, 0:2] + v / sp * (S[ahead, 8:9] + sp * DT * rng.uniform(1.5, 3.5, (40, 1)))
    S[:, 10:12] = G[:, 0]
    return S, G, safety


@functools.lru_cache(maxsize=None)
def _example_crowd():
    from social_navigation_pyenvs_b200 import scenarios
    S, G, safety = _crowd_with_walls(scenarios.EXAMPLE_WALLS, 0.7, seed=7)
    assert S.shape[0] % 128 != 0 and S.shape[0] > 1400  # ragged last tile
    return S, G, safety, scenarios.pack_walls(scenarios.EXAMPLE_WALLS)


def _oracle(model, S, G, walls, safety, k, symmetric=True, numba_compat=False):
    n = S.shape[0]
    cfg = OracleConfig(oracle.type_code(model), False, symmetric, numba_compat)
    params = np.tile(oracle.default_params(model), (1, n, 1))
    ref, Gr, Dr = oracle.update_humans(cfg, S[None], G[None], walls, params, safety[None], np.zeros((1, n, 2)), DT, k, n_threads=8)
    return ref[0], Gr[0], Dr[0]


def _err(got, ref):
    return float(rel_err(wrap_angle_cols(got[:, :8], ref[:, :8]), ref[:, :8]).max())


def _run_against_oracle(model, dtype, S, G, walls, safety, symmetric=True, numba_compat=False):
    """fp64: 3 sub-steps in one call, then 2 in a second, each against the oracle (columns 0-7 relative, current goal exact).
    fp32 (inputs rounded to fp32): one sub-step, then the 3 + 2 run.  Returns the errors {label: max relative error}."""
    from social_navigation_pyenvs_b200.large import LargeCrowd
    if dtype == torch.float32:
        S, G, walls, safety = _f32(S, G, walls, safety)
    kw = dict(walls=walls, dtype=dtype, symmetric=symmetric, numba_compat=numba_compat, safety=safety)
    ref3, G3, D3 = _oracle(model, S, G, walls, safety, 3, symmetric, numba_compat)
    ref5, _, _ = oracle.update_humans(OracleConfig(oracle.type_code(model), False, symmetric, numba_compat), ref3[None], G3[None], walls,
                                      np.tile(oracle.default_params(model), (1, S.shape[0], 1)), safety[None], D3[None], DT, 2, n_threads=8)
    ref5 = ref5[0]
    ref1, _, _ = _oracle(model, S, G, walls, safety, 1, symmetric, numba_compat)
    # the run switches goals on the first sub-step and on later ones
    assert (ref1[:, 10:12] != S[:, 10:12]).any(axis=1).sum() >= 20
    assert (ref5[:, 10:12] != ref1[:, 10:12]).any(axis=1).sum() >= 5
    errs = {}
    if dtype == torch.float32:
        one = LargeCrowd(model, S, G, **kw)
        _step(one, 1)
        got = one.local_rows(S)
        errs["1"] = _err(got, ref1)
        assert np.array_equal(got[:, 10:12], ref1[:, 10:12])
    crowd = LargeCrowd(model, S, G, **kw)
    _step(crowd, 3)
    got3 = crowd.local_rows(S)
    _step(crowd, 2)
    got5 = crowd.local_rows(S)
    errs["3"], errs["5"] = _err(got3, ref3), _err(got5, ref5)
    assert np.array_equal(got3[:, 10:12], ref3[:, 10:12]) and np.array_equal(got5[:, 10:12], ref5[:, 10:12])
    print(f"large parity {model} {str(dtype)[6:]} sym={symmetric} numba={numba_compat}: max rel err " +
          " ".join(f"{k} sub-steps {v:.2e}" for k, v in errs.items()))
    return errs


def _check(model, dtype, errs):
    if dtype == torch.float64:
        tol = 1e-6 if "moussaid" in model else 1e-9
        assert errs["3"] < tol and errs["5"] < tol, (model, errs)
    else:
        # One sub-step: the per-step bar of the bench configurations.  Five: what fp32 rounding accumulates through a crowd --
        # on a B200, at most 1.6e-4 where the torque follows the desired force, but up to 2.3e-3 for the "new" HSFM, whose torque
        # follows the TOTAL force: near force balance its direction, and so the heading, is ill-conditioned.
        bound5 = 5e-3 if model.startswith("hsfm_new") else 5e-4
        assert errs["1"] < 1e-4 and errs["5"] < bound5, (model, errs)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("model", SFMS)
def test_every_model_against_the_oracle(model, dtype):
    """Each model launches its own k_large_finish<T, OBS, HEADED> and pair law: all nine, with the wall group of three, per-human
    safety, goal switches and a ragged last tile."""
    S, G, safety, walls = _example_crowd()
    _check(model, dtype, _run_against_oracle(model, dtype, S, G, walls, safety))


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
def test_numba_compat_semantics(dtype):
    """numba_compat with hsfm_guo and walls: Guo wall force divided by W, first-wins closest segment, '<=' goal test, zero desired
    force inside the goal radius.  One human stands exactly on its goal, one exactly at its radius from it (dg == r)."""
    S, G, safety, walls = _example_crowd()
    S, G = S.copy(), G.copy()
    i, j = 5, 6
    for h in (i, j):
        S[h, 0:2] = np.round(S[h, 0:2] * 64) / 64  # exact in fp32 too
    G[i, 0] = S[i, 0:2]
    S[j, 8] = 0.25
    G[j, 0] = S[j, 0:2] + [0.25, 0.0]
    S[:, 10:12] = G[:, 0]
    _check("hsfm_guo", dtype, _run_against_oracle("hsfm_guo", dtype, S, G, walls, safety, numba_compat=True))


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("model", ["sfm_moussaid", "hsfm_new_moussaid"])
def test_asymmetric_pair_order(model, dtype):
    """symmetric=False: every pair evaluated in the agent's own order (no swap of the Moussaid pair law in pairs_chunk)."""
    S, G, safety, walls = _example_crowd()
    _check(model, dtype, _run_against_oracle(model, dtype, S, G, walls, safety, symmetric=False))


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
def test_wall_set_beyond_48_kb_of_shared_memory(dtype):
    """24 polygons of 30 segments: 720 staged segments, 51 KB of dynamic shared memory in fp64 with the exp table -- the finish
    kernel is launched after raising its shared-memory limit."""
    from social_navigation_pyenvs_b200 import scenarios
    a = np.linspace(0.0, 2 * np.pi, 30, endpoint=False)
    centres = [(x, y) for x in (-15.5, -9.5, -3.5, 2.5, 8.5, 14.5) for y in (-12.5, -4.5, 3.5, 11.5)]
    polygons = [[[cx + 0.6 * np.cos(t), cy + 0.6 * np.sin(t)] for t in a] for cx, cy in centres]
    walls = scenarios.pack_walls(polygons)
    assert walls.shape[:2] == (24, 30) and 16384 + 48 * 24 * 30 > 48 * 1024  # fp64: exp table + 48 bytes per segment
    S, G, safety = _crowd_with_walls(polygons, 0.8, seed=9)
    _check("hsfm_new_guo", dtype, _run_against_oracle("hsfm_new_guo", dtype, S, G, walls, safety))


# ---- slices of one crowd: bit for bit ----

@functools.lru_cache(maxsize=None)
def _grid72(order):
    from social_navigation_pyenvs_b200 import scenarios
    sc = scenarios.jittered_grid_crowd(72, pitch=1.0, jitter=0.3, seed=3)
    S, G = sc["states"][0], sc["goals"][0]
    if order == "patch":
        perm = scenarios.spatial_order(S[:, 0:2])
        S, G = np.ascontiguousarray(S[perm]), np.ascontiguousarray(G[perm])
    S[:, 5:7] = np.random.RandomState(1).uniform(-0.6, 0.6, (S.shape[0], 2))
    return S, G


@functools.lru_cache(maxsize=None)
def _whole_after_one(order, model, dtype):
    from social_navigation_pyenvs_b200.large import LargeCrowd
    S, G = _grid72(order)
    crowd = LargeCrowd(model, S, G, dtype=dtype, symmetric=True)
    _step(crowd, 1)
    return crowd.local_rows(S)


N72 = 72 * 72
SLICES = [(0, 1000), (128, 700), (3968, 1), (0, 100), (64, N72 - 64), (N72 - 1000, 1000), (1024, 1024)]


@pytest.mark.parametrize("shard", SLICES, ids=[f"{o}+{n}" for o, n in SLICES])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("model", ["hsfm_farina", "hsfm_new_guo"])
@pytest.mark.parametrize("order", ["row", "patch"])
def test_slices_same_bits_as_the_whole_crowd(order, model, dtype, shard):
    """A shard= slice stepped against the frozen rest of the 72 x 72 crowd.  After one sub-step its rows are the whole crowd's
    rows bit for bit (same view, chunks added in ascending order on the work list, the static grid or all pairs), culled and all
    pairs alike; after a second call of two sub-steps culled == all pairs == three calls of one.  A slice that starts on a tile
    takes the work list, whose i-block box comes from the tile boxes: when its last tile also holds other humans, a listed chunk
    can be culled tile by tile against the slice's own agents and must still write its partial sums."""
    from social_navigation_pyenvs_b200.large import LargeCrowd
    S, G = _grid72(order)
    off, n = shard
    rows = S[off:off + n]
    whole = _whole_after_one(order, model, dtype)[off:off + n]
    out = {}
    for cull in (True, False):
        crowd = LargeCrowd(model, S, G, dtype=dtype, symmetric=True, shard=shard)
        crowd.culling = cull
        _step(crowd, 1, whole=False)
        first = crowd.local_rows(rows)
        _step(crowd, 2, whole=False)
        out[cull] = (first, crowd.local_rows(rows))
    single = LargeCrowd(model, S, G, dtype=dtype, symmetric=True, shard=shard)
    for _ in range(3):
        _step(single, 1, whole=False)
    single = single.local_rows(rows)
    assert np.isfinite(out[True][0]).all() and np.isfinite(out[True][1]).all()
    assert np.array_equal(out[True][0], whole), "culled slice != whole crowd after one sub-step"
    assert np.array_equal(out[False][0], whole), "all-pairs slice != whole crowd after one sub-step"
    assert np.array_equal(out[True][1], out[False][1]), "culled != all pairs after a call of two sub-steps"
    assert np.array_equal(out[True][1], single), "2 sub-steps in one call != one per call"


# ---- the culling reach ----

def _reach_probe(model, dtype, inside):
    """129 humans: tile 0 a 16 x 8 patch (pitch 0.8 m, r+s = 0.35) whose right column is at x = 0 with one human at y = 0;
    human 128 alone in tile 1, at rest on the only goal of its list, r+s = 0.32, on the x axis at 1 cm inside or outside
    reach = 0.35 + 0.32 + margin from tile 0's box (margin 700 max(B, D) in fp64, 88 max(B, D) in fp32; D only for Guo)."""
    p = oracle.default_params(model)
    soc = oracle.type_code(model) % 3
    bmax = max(p[3], p[7]) if soc == 1 else p[3]
    f = np.float64 if dtype == torch.float64 else np.float32
    margin = f((700.0 if dtype == torch.float64 else 88.0) * bmax)
    S = np.zeros((129, 13))
    c, r = np.meshgrid(np.arange(16), np.arange(8), indexing="ij")
    S[:128, 0] = -0.8 * (15 - c.ravel())
    S[:128, 1] = 0.8 * (r.ravel() - 4)
    S[:, 8], S[:, 9], S[:, 12] = 0.3, 75.0, 1.0
    safety = np.full(129, 0.05)
    safety[128] = 0.02
    rs0, rs1 = f(f(0.3) + f(0.05)), f(f(0.3) + f(0.02))
    reach = f(f(rs1 + rs0) + margin)  # as the kernel forms it (the i-block's r+s + the tile's + the margin)
    S[128, 0] = float(reach) + (-0.01 if inside else 0.01)
    G = np.zeros((129, 1, 2))
    G[:128, 0] = S[:128, 0:2] + [-5.0, 0.0]
    G[128, 0] = S[128, 0:2]
    S[:, 10:12] = G[:, 0]
    if dtype == torch.float32:
        S, G, safety = _f32(S, G, safety)
    return S, G, safety, p, soc, bmax


@pytest.mark.parametrize("inside", [True, False], ids=["inside", "outside"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("model", ["sfm_helbing", "hsfm_farina", "sfm_guo", "hsfm_new_guo"])
def test_culling_reach_boundary(model, dtype, inside):
    """1 cm inside the reach the tile is evaluated: culled == all pairs bit for bit and the lone human moves (in fp32 by a
    subnormal few 1e-39 m/s -- nothing flushes it).  1 cm outside it culling leaves the human exactly at rest, and all pairs moves it
    by no more than the pair law allows there: sum_j A e^((r_ij - d_ij)/B) + C e^((r_ij - d_ij)/D) times dt/m (x2 for the HSFM
    body frame), where in fp64 every pair also counts at least 2^-1009 (the exponent clamp of exp2_scaled_times)."""
    from social_navigation_pyenvs_b200.large import LargeCrowd
    S, G, safety, p, soc, bmax = _reach_probe(model, dtype, inside)
    out = {}
    for cull in (True, False):
        crowd = LargeCrowd(model, S, G, dtype=dtype, symmetric=True, safety=safety)
        crowd.culling = cull
        _step(crowd, 1)
        out[cull] = crowd.local_rows(S)
    dv = {cull: np.hypot(out[cull][128, 3], out[cull][128, 4]) for cull in out}
    if inside:
        assert np.array_equal(out[True], out[False])
        assert dv[True] > 0.0, "the tile in reach was not evaluated"
        return
    assert np.array_equal(out[True][128, :8], S[128, :8]), "a culled tile moved the human"
    d = np.hypot(S[:128, 0] - S[128, 0], S[:128, 1] - S[128, 1])
    x = (S[:128, 8] + safety[:128] + S[128, 8] + safety[128]) - d
    pair = p[1] * np.exp(x / p[3]) + (p[5] * np.exp(x / p[7]) if soc == 1 else 0.0)
    assert x.max() < -(88 if dtype == torch.float32 else 700) * bmax
    if dtype == torch.float64:
        pair = np.maximum(pair, 2.0 ** -1009)
    bound = 2.0 * pair.sum() * DT / S[128, 9]
    assert dv[False] <= bound, (float(dv[False]), bound)
