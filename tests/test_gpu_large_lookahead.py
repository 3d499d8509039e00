"""The policies' one-step lookahead (snp_lookahead, crowd_nav/policy/cadrl.py:42-83) for envs whose humans do not fit one CTA's
shared memory (fp64 N > 673, > 609 with theta and omega visible; fp32 N > 1312 / > 1190): the humans of an env are split into
chunks of 256 over several CTAs and the swept test's rewards folded across the chunks.

* the oracle beyond each threshold, through TiledCrowdEngine.lookahead(query_env=False) and lookahead_from(the state of a stepped
  engine), with the deciding human in the first, a middle and the last (ragged) chunk and a collision in one chunk while the
  smallest non-negative distance lies in another; every output word written (NaN fill);
* the split equal to the whole-env kernel bit for bit where both run, with bulk copies and with vector stores;
* one crowd of 65 536 humans, and a batch of more than 2^31 output words."""
import numpy as np
import pytest
import torch

import oracle
from helpers import rel_err
from test_gpu_block_packed import THREADS, _look_batch
from test_gpu_lookahead import _actions, _oracle_inputs

pytestmark = pytest.mark.gpu

DT = 0.25
MODELS = ["hsfm_farina", "sfm_guo", "sfm_helbing"]
CHUNK = 256  # humans per CTA of the split (kLookThreads)


def _one_cta_holds(N, visible, itemsize):
    """launch_lookahead's whole-env layout with one action per CTA fits 200 KB (csrc/snp_lookahead.cu LookSmem)."""
    r16 = lambda x: (x + 15) & ~15
    off = r16(r16(r16(itemsize * 11 * N) + 16 + 8 * itemsize) + 8 * N)
    return off + 2 * r16(N * (15 if visible else 13) * itemsize + 16) <= 200 * 1024


def test_one_cta_thresholds():
    """The largest N one CTA holds, per dtype and row width (the sizes of the parity test straddle them)."""
    last = lambda vis, size: max(n for n in range(1, 2000) if _one_cta_holds(n, vis, size))
    assert (last(False, 8), last(True, 8), last(False, 4), last(True, 4)) == (673, 609, 1312, 1190)


def _scene(E, N, seed):
    """_look_batch's robots (near the goal, 0.05 m and 0.15 m from a human at rest, alone) with the deciding human moved to the
    first (index 3), a middle (N // 2) or the last chunk (N - 2) by env; env 1 gets a second human at rest 0.15 m from its robot on
    the other side, in the first chunk: actions towards one of the two collide in its chunk while the other's chunk holds the
    smallest non-negative distance."""
    S, G, R = _look_batch(E, N, seed)
    for e in range(E):
        if e % 4 not in (1, 2):
            continue
        h = int(np.argmin(np.hypot(*(S[e, :, 0:2] - R[e, 0:2]).T)))
        t = (3, N // 2, N - 2)[e % 3]
        S[e, [h, t]], G[e, [h, t]] = S[e, [t, h]], G[e, [t, h]]
    h, b = N // 2, 3
    u = (S[1, h, 0:2] - R[1, 0:2]) / np.hypot(*(S[1, h, 0:2] - R[1, 0:2]))
    S[1, b, 0:2] = R[1, 0:2] - (0.3 + S[1, b, 8] + 0.15) * u
    S[1, b, 3:5] = 0.0
    return S, G, R


def _inputs(eng, nxt, vis, sel=slice(None), yaw_from_next=False):
    cur, nxo, rob = _oracle_inputs(eng, nxt, vis, sel)
    if vis and yaw_from_next and not eng.headed:  # the constant-velocity propagation integrates the yaw of every model
        from social_navigation_pyenvs_b200 import _lib as L
        nx = nxt.double().cpu().numpy()[:, sel]
        nxo[..., 2], nxo[..., 5] = nx[L.DYN_TH], nx[L.DYN_OM]
    return cur, nxo, rob


def _check(rot, rew, eng, nxt, vis, dtype, sel=slice(None), yaw_from_next=False, kinds=True):
    cur, nxo, rob = _inputs(eng, nxt, vis, sel, yaw_from_next)
    rot_ref, rew_ref = oracle.lookahead(cur, nxo, rob, _actions(), DT, visible=vis, n_threads=THREADS)
    idx = torch.as_tensor(np.arange(eng.E)[sel], device=rew.device)
    assert np.array_equal(rew[idx].cpu().numpy(), rew_ref)
    err = rel_err(rot[idx].double().cpu().numpy(), rot_ref).max()
    assert err < (1e-9 if dtype == torch.float64 else 1e-4), err
    if kinds:
        assert (rew_ref == -0.25).any() and (rew_ref == 1.0).any() and ((rew_ref < 0) & (rew_ref > -0.25)).any() and (rew_ref == 0).any()


def _nan(eng):
    eng._rotated.fill_(float("nan")); eng._rewards.fill_(float("nan"))


def _written(rot, rew):
    assert not torch.isnan(rot).any() and not torch.isnan(rew).any()


@pytest.mark.parametrize("visible", [False, True], ids=["hidden", "visible"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("N", [610, 674, 1000, 1024, 1191, 1313, 4096])
def test_lookahead_vs_oracle_beyond_one_cta(N, dtype, visible):
    """E = 8 envs: TiledCrowdEngine.lookahead(query_env=False) and lookahead_from(next = the humans of a copy stepped 20 sub-steps),
    each on outputs filled with NaN; rewards bit-exact and rotated states within 1e-9 / 1e-4 of the oracle on the engine's state."""
    from social_navigation_pyenvs_b200 import TiledCrowdEngine
    E = 8
    model = MODELS[[610, 674, 1000, 1024, 1191, 1313, 4096].index(N) % 3]
    S, G, R = _scene(E, N, 7100 + N)
    make = lambda: TiledCrowdEngine.from_reference_arrays(model, S, G, consider_robot=False, all_params_equal=True, robot=R, dtype=dtype)
    eng = make()
    eng.set_action_space(_actions())
    eng.lookahead(DT, theta_and_omega_visible=visible, query_env=False)
    _nan(eng)
    rot, rew = eng.lookahead(DT, theta_and_omega_visible=visible, query_env=False)
    _written(rot, rew)
    _check(rot, rew, eng, eng._peek_buf, visible, dtype, yaw_from_next=True)

    stepped = make()
    stepped.update_humans(dt=0.0125, n_substeps=20)
    _nan(eng)
    rot, rew = eng.lookahead_from(stepped.dyn, DT, theta_and_omega_visible=visible)
    _written(rot, rew)
    _check(rot, rew, eng, stepped.dyn, visible, dtype)


def _same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("N,dtype,visible", [(n, d, v) for n in (25, 300, 512) for d in (torch.float64, torch.float32) for v in (False, True)]
                         + [(673, torch.float64, False)])
def test_split_equals_one_cta_bit_for_bit(N, dtype, visible):
    """split_humans=True against the whole-env kernel, rotated states and rewards, with bulk copies and with vector stores; N = 673 is
    the largest fp64 13-value env one CTA holds."""
    from social_navigation_pyenvs_b200 import CrowdEngine
    E = 8
    S, G, R = _scene(E, N, 7300 + N)
    eng = CrowdEngine.from_reference_arrays("hsfm_farina", S, G, consider_robot=False, all_params_equal=True, robot=R, dtype=dtype)
    eng.set_action_space(_actions())
    nxt = eng.constant_velocity_next(DT)
    assert _one_cta_holds(N, visible, 8 if dtype == torch.float64 else 4)
    ref = [t.clone() for t in eng.lookahead_from(nxt, DT, theta_and_omega_visible=visible, yaw_from_next=True)]
    for bulk in (True, False):
        one = [t.clone() for t in eng.lookahead_from(nxt, DT, theta_and_omega_visible=visible, yaw_from_next=True, bulk_store=bulk)]
        _nan(eng)
        split = eng.lookahead_from(nxt, DT, theta_and_omega_visible=visible, yaw_from_next=True, bulk_store=bulk, split_humans=True)
        assert _same(one, ref) and _same(split, ref), bulk
    if N > CHUNK:
        _check(*split, eng, nxt, visible, dtype, yaw_from_next=True)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
def test_vector_stores_beyond_one_cta(dtype):
    """The split's vector-store fallback writes the same bits as its bulk copies (N = 1313, ragged last chunk)."""
    from social_navigation_pyenvs_b200 import TiledCrowdEngine
    E, N = 4, 1313
    S, G, R = _scene(E, N, 7500)
    eng = TiledCrowdEngine.from_reference_arrays("sfm_guo", S, G, consider_robot=False, all_params_equal=True, robot=R, dtype=dtype)
    eng.set_action_space(_actions())
    nxt = eng.constant_velocity_next(DT)
    for vis in (False, True):
        bulk = [t.clone() for t in eng.lookahead_from(nxt, DT, theta_and_omega_visible=vis, yaw_from_next=True)]
        _nan(eng)
        assert _same(eng.lookahead_from(nxt, DT, theta_and_omega_visible=vis, yaw_from_next=True, bulk_store=False), bulk), vis


def test_one_crowd_of_65536_humans():
    """TiledCrowdEngine(E = 1), N = 65 536, fp64 (552 MB of rotated states): the whole output against the oracle, with two humans
    next to the robot in the first and a middle chunk (_scene's env 1)."""
    from social_navigation_pyenvs_b200 import TiledCrowdEngine
    N = 65536
    S, G, R = (x[1:2] for x in _scene(2, N, 7700))
    eng = TiledCrowdEngine.from_reference_arrays("hsfm_farina", S, G, consider_robot=False, all_params_equal=True, robot=R)
    eng.set_action_space(_actions())
    eng.lookahead(DT, query_env=False)
    _nan(eng)
    rot, rew = eng.lookahead(DT, query_env=False)
    _written(rot, rew)
    _check(rot, rew, eng, eng._peek_buf, False, torch.float64, yaw_from_next=True, kinds=False)
    r = rew.cpu().numpy()
    assert (r == -0.25).any() and ((r < 0) & (r > -0.25)).any()


def test_output_of_more_than_2_31_words():
    """E = 64, N = 32 768, fp32, 13 values: 2.2e9 words (8.8 GB).  No NaN left; the oracle on sampled envs including the last."""
    from social_navigation_pyenvs_b200 import TiledCrowdEngine
    E, N = 64, 32768
    S, G, R = _scene(E, N, 7900)
    eng = TiledCrowdEngine.from_reference_arrays("sfm_helbing", S, G, consider_robot=False, all_params_equal=True, robot=R,
                                                 dtype=torch.float32)
    del S, G
    eng.set_action_space(_actions())
    eng.lookahead(DT, query_env=False)
    assert eng._rotated.numel() > 2 ** 31
    _nan(eng)
    rot, rew = eng.lookahead(DT, query_env=False)
    _written(rot, rew)
    for e in (1, 2, 33, E - 1):
        _check(rot, rew, eng, eng._peek_buf, False, torch.float32, sel=[e], yaw_from_next=True, kinds=False)
