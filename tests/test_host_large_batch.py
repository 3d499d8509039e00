"""CPU-side checks of snp_large_batch_step (E environments through the tiled kernels): what it does not implement and bad arguments
are refused before anything touches the device (the pointers are dummies), and its scratch covers every region."""
import ctypes

import pytest

DUMMY = ctypes.c_void_p(4096)
E, N = 3, 700


def _crowd(L, robot=True, **kw):
    args = dict(E=E, N=N, G=2, dtype=L.SNP_F64, dyn=DUMMY, stat=DUMMY, goals=DUMMY, goal_idx=DUMMY, goal_cnt=DUMMY, robot=DUMMY if robot else None)
    args.update(kw)
    return L.SnpCrowd(**args)


def _opts(L):
    return L.SnpStepOpts(type=3, dt=0.0125, n_substeps=2, consider_robot=1, robot_mode=1, action=DUMMY, flags=DUMMY, checks=DUMMY,
                         pre_checks=1, post_checks=1)


def _run(L, c, o, n_bytes=None, scratch=DUMMY):
    lib = L.lib()
    if n_bytes is None:
        n_bytes = int(lib.snp_large_batch_scratch_bytes(E, N, L.SNP_F64))
    opts = None if o is None else ctypes.byref(o)
    return lib.snp_large_batch_step(ctypes.byref(c), opts, scratch, n_bytes, None)


@pytest.mark.parametrize("option", ["robot_mode2", "robot_every", "track_touch", "post_checks2", "dyn_out", "respawn", "agent_params"])
def test_batch_step_refuses_unsupported_options_before_any_launch(option):
    from social_navigation_pyenvs_b200 import _lib as L
    c, o = _crowd(L), _opts(L)
    if option == "robot_mode2":
        o.robot_mode = 2
    elif option == "robot_every":
        o.robot_every = 2
    elif option == "post_checks2":
        o.post_checks = 2
    elif option == "dyn_out":
        o.dyn_out = DUMMY
    elif option == "agent_params":
        c = _crowd(L, agent_params=DUMMY)
    else:
        setattr(o, option, 1)
    assert _run(L, c, o) == -3, option
    assert "snp_large_batch_step" in L.lib().snp_last_error().decode()


@pytest.mark.parametrize("case", ["null_opts", "null_scratch", "E0", "N0", "G0", "dtype", "type9", "no_dyn", "no_goal_cnt", "walls_no_array",
                                  "negative_substeps", "mode4", "mode_negative", "no_robot_visible", "no_robot_moving", "no_robot_checks",
                                  "no_action_moving", "no_action_pre", "no_flags", "scratch_short", "scratch_misaligned"])
def test_batch_step_refuses_bad_arguments_before_any_launch(case):
    from social_navigation_pyenvs_b200 import _lib as L
    lib = L.lib()
    c, o = _crowd(L), _opts(L)
    n_bytes, scratch = int(lib.snp_large_batch_scratch_bytes(E, N, L.SNP_F64)), DUMMY
    if case == "null_opts":
        o = None
    elif case == "null_scratch":
        scratch = None
    elif case in ("E0", "N0", "G0"):
        c = _crowd(L, **{case[0]: 0})
    elif case == "dtype":
        c = _crowd(L, dtype=7)
    elif case == "type9":
        o.type = 9
    elif case == "no_dyn":
        c = _crowd(L, dyn=None)
    elif case == "no_goal_cnt":
        c = _crowd(L, goal_cnt=None)
    elif case == "walls_no_array":
        c = _crowd(L, W=2, S=4)
    elif case == "negative_substeps":
        o.n_substeps = -1
    elif case == "mode4":
        o.robot_mode = 4
    elif case == "mode_negative":
        o.robot_mode = -1
    elif case == "no_robot_visible":
        c, o.robot_mode, o.pre_checks, o.post_checks = _crowd(L, robot=False), 0, 0, 0
    elif case == "no_robot_moving":
        c, o.consider_robot, o.pre_checks, o.post_checks = _crowd(L, robot=False), 0, 0, 0
    elif case == "no_robot_checks":
        c, o.consider_robot, o.robot_mode, o.pre_checks = _crowd(L, robot=False), 0, 0, 0
    elif case == "no_action_moving":
        o.action, o.pre_checks = None, 0
    elif case == "no_action_pre":
        o.action, o.robot_mode = None, 0
    elif case == "no_flags":
        o.flags = None
    elif case == "scratch_short":
        n_bytes -= 1
    elif case == "scratch_misaligned":
        scratch = ctypes.c_void_p(4096 + 8)
    assert _run(L, c, o, n_bytes, scratch) == -1, case
    assert "snp_large_batch_step" in lib.snp_last_error().decode()


def test_batch_scratch_size_covers_every_region():
    """snp_large_batch_scratch_bytes is host arithmetic: the partial sums [J][2][E N] with J = ceil(N/128) chunks per env, the live
    map and the lists of E ceil(N/128) i-blocks, the queue counters, then two view buffers of [5][E N] entities and [E ceil(N/128)][5]
    tile boxes -- for whole and ragged N and both dtypes (at most 15 bytes of alignment per region)."""
    from social_navigation_pyenvs_b200 import _lib as L
    lib = L.lib()
    for E_, N_ in ((64, 1024), (16, 4096), (4, 16384), (5, 513), (5, 1000), (1, 1), (3, 300)):
        for dtype, w in ((L.SNP_F64, 8), (L.SNP_F32, 4)):
            J = -(-N_ // 128)
            blocks, Jp = E_ * J, (J + 15) // 16 * 16
            views = 2 * w * 5 * (E_ * N_ + E_ * J)
            need = w * J * 2 * E_ * N_ + blocks * Jp + 4 * (260 + blocks * J + blocks + blocks * Jp) + views
            got = int(lib.snp_large_batch_scratch_bytes(E_, N_, dtype))
            assert need <= got <= need + 7 * 16, (E_, N_, dtype, need, got)
    for bad in ((0, 10, L.SNP_F64), (2, 0, L.SNP_F64), (2, 10, 7)):
        assert int(lib.snp_large_batch_scratch_bytes(*bad)) == -1, bad


def test_the_engine_refuses_what_the_tiled_path_does_not_have():
    """TiledCrowdEngine's peek, lookahead through it, imitation_learning_step, sim_update and step_host raise without a device."""
    from social_navigation_pyenvs_b200 import TiledCrowdEngine
    eng = TiledCrowdEngine.__new__(TiledCrowdEngine)
    for call in (lambda: eng.peek(0.25), lambda: eng.imitation_learning_step(), lambda: eng.sim_update(), lambda: eng.step_host(None, None, None, None),
                 lambda: eng.get_next_human_observable_states(0.25)):
        with pytest.raises(NotImplementedError, match="TiledCrowdEngine"):
            call()
