"""CPU-side checks of the large crowd's robot: snp_large_run_p2p refuses what it does not implement, and snp_large_checks refuses bad
arguments, before anything touches the device (the pointers are dummies); the robot needs no scratch."""
import ctypes

import pytest

DUMMY = ctypes.c_void_p(4096)


def _crowd(L, robot=True, dtype=None):
    return L.SnpCrowd(E=1, N=256, G=2, dtype=L.SNP_F64 if dtype is None else dtype, dyn=DUMMY, stat=DUMMY, goals=DUMMY, goal_idx=DUMMY,
                      goal_cnt=DUMMY, robot=DUMMY if robot else None)


def _run(L, c, o):
    lib = L.lib()
    views = (ctypes.c_void_p * 1)(4096)
    n_bytes = int(lib.snp_large_scratch_bytes(256, 256, L.SNP_F64))
    return lib.snp_large_run_p2p(ctypes.byref(c), ctypes.byref(o), views, views, 0, 256, 0, 1, 0, views, 0, 1, DUMMY, DUMMY, n_bytes, None)


@pytest.mark.parametrize("option", ["robot_mode2", "track_touch", "pre_checks", "post_checks", "dyn_out", "respawn"])
def test_large_step_rejects_unsupported_options_before_any_launch(option):
    from social_navigation_pyenvs_b200 import _lib as L
    o = L.SnpStepOpts(type=3, dt=0.0125, consider_robot=1, robot_mode=1, action=DUMMY)
    if option == "robot_mode2":
        o.robot_mode = 2
    elif option == "dyn_out":
        o.dyn_out = DUMMY
    else:
        setattr(o, option, 1)
    assert _run(L, _crowd(L), o) == -3, option
    msg = L.lib().snp_last_error().decode()
    assert "snp_large_run_p2p" in msg
    if option in ("pre_checks", "post_checks"):
        assert "snp_large_checks" in msg


@pytest.mark.parametrize("case", ["no_robot_visible", "no_robot_moving", "no_action", "mode4", "mode_negative"])
def test_large_step_rejects_an_incomplete_robot_before_any_launch(case):
    from social_navigation_pyenvs_b200 import _lib as L
    c, o = _crowd(L), L.SnpStepOpts(type=0, dt=0.0125, action=DUMMY)
    if case == "no_robot_visible":
        c, o.consider_robot = _crowd(L, robot=False), 1
    elif case == "no_robot_moving":
        c, o.robot_mode = _crowd(L, robot=False), 3
    elif case == "no_action":
        o.robot_mode, o.action = 1, None
    elif case == "mode4":
        o.robot_mode = 4
    else:
        o.robot_mode = -1
    assert _run(L, c, o) == -1, case
    assert "snp_large_run_p2p" in L.lib().snp_last_error().decode()


@pytest.mark.parametrize("case", ["null_view", "null_radius", "null_opts", "M0", "no_robot", "no_flags", "no_action", "nothing", "dtype",
                                  "mode2", "post2"])
def test_large_checks_rejects_bad_arguments_before_any_launch(case):
    from social_navigation_pyenvs_b200 import _lib as L
    lib = L.lib()
    c = _crowd(L)
    o = L.SnpStepOpts(type=0, dt=0.0125, action=DUMMY, flags=DUMMY, pre_checks=1, post_checks=1)
    view, radius, M, expect = DUMMY, DUMMY, 256, -1
    if case == "null_view":
        view = None
    elif case == "null_radius":
        radius = None
    elif case == "M0":
        M = 0
    elif case == "no_robot":
        c = _crowd(L, robot=False)
    elif case == "no_flags":
        o.flags = None
    elif case == "no_action":
        o.action = None
    elif case == "nothing":
        o.pre_checks = o.post_checks = 0
    elif case == "dtype":
        c = _crowd(L, dtype=7)
    elif case == "mode2":
        o.robot_mode = 2
    elif case == "post2":
        o.post_checks, expect = 2, -3
    opts = None if case == "null_opts" else ctypes.byref(o)
    assert lib.snp_large_checks(ctypes.byref(c), opts, view, radius, M, None) == expect, case
    assert "snp_large_checks" in lib.snp_last_error().decode()


def test_large_scratch_size_is_unchanged_by_the_robot():
    """The robot is recomputed by every thread from crowd->robot: no scratch region of its own.  Sizes pinned at the values before
    the robot existed."""
    from social_navigation_pyenvs_b200 import _lib as L
    lib = L.lib()
    got = [int(lib.snp_large_scratch_bytes(n, M, d)) for n, M in ((65536, 65536), (8192, 65536), (1517, 1517), (500, 500))
           for d in (L.SNP_F64, L.SNP_F32)]
    assert got == [539233296, 270797840, 67405072, 33850640, 293888, 148256, 33440, 17440]
