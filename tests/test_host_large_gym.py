"""CPU-side checks of the gym beyond 512 humans per env: snp_reset refuses crowds its CTA kernel cannot hold before anything touches
the device (the pointers are dummies), the Python bit matches the header, and the gym picks the tiled engine above 512 humans."""
import ctypes
import os

import pytest

DUMMY = ctypes.c_void_p(4096)
CTA_LIMIT = (200 * 1024 - 624 * 4) // 32  # 624 generator words + x, y, r, vd per human in 200 KB of shared memory


def _reset(L, N, reserved=0):
    c = L.SnpCrowd(E=2, N=N, G=2, dtype=L.SNP_F64, dyn=DUMMY, stat=DUMMY, goals=DUMMY, goal_idx=DUMMY, goal_cnt=DUMMY, robot=DUMMY)
    g = L.SnpResetArgs(scenario=0, circle_radius=7.0, robot_radius=0.3, traffic_length=14.0, traffic_height=3.0, reserved=reserved)
    return L.lib().snp_reset(ctypes.byref(c), ctypes.byref(g), None)


@pytest.mark.parametrize("N,reserved", [(CTA_LIMIT + 1, 0), (CTA_LIMIT + 1, 1), (20000, 0)])
def test_reset_refuses_crowds_beyond_the_cta_kernel_before_any_launch(N, reserved):
    from social_navigation_pyenvs_b200 import _lib as L
    assert _reset(L, N, reserved) == -3
    msg = L.lib().snp_last_error().decode()
    assert f"{N} humans per env" in msg and f"at most {CTA_LIMIT}" in msg


def test_reset_force_cta_bit_matches_the_header():
    from social_navigation_pyenvs_b200 import _lib as L
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "include", "snp_b200.h")) as f:
        assert f"SNP_RESET_FORCE_CTA = {L.SNP_RESET_FORCE_CTA} " in f.read()


@pytest.mark.parametrize("n,tiled", [(5, False), (512, False), (513, True), (4096, True)])
def test_gym_runs_above_512_humans_on_the_tiled_engine(n, tiled):
    from social_navigation_pyenvs_b200 import CrowdEngine, TiledCrowdEngine
    from social_navigation_pyenvs_b200.social_nav_gym import BatchedSocialNavGym
    g = BatchedSocialNavGym(2, device="cpu")
    g.configure(dict(human_num=n))
    assert g._engine_class() is (TiledCrowdEngine if tiled else CrowdEngine)
    assert g.spatial_order
