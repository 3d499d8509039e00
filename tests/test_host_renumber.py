"""CPU-side checks of the re-numbering entries (snp_spatial_order, snp_gather_crowd, snp_large_tile_boxes): null and bad arguments are
refused before anything touches the device (the pointers are dummies), and a crowd stepped as a slice against a frozen rest
(LargeCrowd(shard=...)) cannot be re-numbered."""
import ctypes

import pytest

DUMMY = ctypes.c_void_p(4096)


def _order(L, case):
    args = dict(px=DUMMY, py=DUMMY, E=2, N=256, dtype=L.SNP_F64, world=1, perm=DUMMY, nonfinite=DUMMY, scratch=DUMMY, nbytes=1 << 30)
    if case.startswith("null_"):
        args[case[5:]] = None
    elif case == "E0":
        args["E"] = 0
    elif case == "N0":
        args["N"] = 0
    elif case == "too_many":
        args["E"], args["N"] = 1 << 16, 1 << 15
    elif case == "dtype":
        args["dtype"] = 7
    elif case == "world0":
        args["world"] = 0
    elif case == "deal_ragged":
        args["world"], args["N"] = 2, 200
    elif case == "scratch_misaligned":
        args["scratch"] = ctypes.c_void_p(4096 + 8)
    return L.lib().snp_spatial_order(*args.values(), None)


@pytest.mark.parametrize("case", ["null_px", "null_py", "null_perm", "null_nonfinite", "null_scratch", "E0", "N0", "too_many", "dtype",
                                  "world0", "deal_ragged", "scratch_misaligned"])
def test_spatial_order_refuses_bad_arguments_before_any_launch(case):
    from social_navigation_pyenvs_b200 import _lib as L
    assert _order(L, case) == -1, case
    assert "snp_spatial_order" in L.lib().snp_last_error().decode()


def test_spatial_order_scratch_size_refuses_bad_sizes():
    from social_navigation_pyenvs_b200 import _lib as L
    for E, N in ((0, 10), (2, 0), (1 << 16, 1 << 15)):
        assert int(L.lib().snp_spatial_order_scratch_bytes(E, N)) == -1, (E, N)
        assert "snp_spatial_order_scratch_bytes" in L.lib().snp_last_error().decode()


def _crowd(L, **kw):
    args = dict(E=2, N=256, G=2, dtype=L.SNP_F64, dyn=DUMMY, stat=DUMMY, goals=DUMMY, goal_idx=DUMMY, goal_cnt=DUMMY)
    args.update(kw)
    return L.SnpCrowd(**args)


@pytest.mark.parametrize("case", ["null_dst", "null_src", "null_perm", "dst_no_dyn", "src_no_goal_cnt", "dtype_mismatch", "dtype_bad", "E_mismatch",
                                  "E0", "G_mismatch", "N0", "slice_past_end", "negative_offset", "agent_params"])
def test_gather_crowd_refuses_bad_arguments_before_any_launch(case):
    from social_navigation_pyenvs_b200 import _lib as L
    dst, src, perm, offset = _crowd(L, N=128), _crowd(L, N=512), DUMMY, 0
    if case == "dst_no_dyn":
        dst = _crowd(L, N=128, dyn=None)
    elif case == "src_no_goal_cnt":
        src = _crowd(L, N=512, goal_cnt=None)
    elif case == "dtype_mismatch":
        src = _crowd(L, N=512, dtype=L.SNP_F32)
    elif case == "dtype_bad":
        dst, src = _crowd(L, N=128, dtype=7), _crowd(L, N=512, dtype=7)
    elif case == "E_mismatch":
        src = _crowd(L, N=512, E=3)
    elif case == "E0":
        dst, src = _crowd(L, N=128, E=0), _crowd(L, N=512, E=0)
    elif case == "G_mismatch":
        src = _crowd(L, N=512, G=1)
    elif case == "N0":
        dst = _crowd(L, N=0)
    elif case == "slice_past_end":
        offset = 512 - 127
    elif case == "negative_offset":
        offset = -1
    elif case == "agent_params":
        dst = _crowd(L, N=128, agent_params=DUMMY)
    elif case == "null_perm":
        perm = None
    rc = L.lib().snp_gather_crowd(None if case == "null_dst" else ctypes.byref(dst), None if case == "null_src" else ctypes.byref(src), perm,
                                  offset, None, None)
    assert rc == (-3 if case == "agent_params" else -1), case
    assert "snp_gather_crowd" in L.lib().snp_last_error().decode()


@pytest.mark.parametrize("case", ["null_view", "M0", "dtype"])
def test_tile_boxes_refuse_bad_arguments_before_any_launch(case):
    from social_navigation_pyenvs_b200 import _lib as L
    view, M, dtype = (None if case == "null_view" else DUMMY), (0 if case == "M0" else 1000), (7 if case == "dtype" else L.SNP_F64)
    assert L.lib().snp_large_tile_boxes(view, M, dtype, None) == -1, case
    assert "snp_large_tile_boxes" in L.lib().snp_last_error().decode()


def test_a_slice_against_a_frozen_rest_cannot_be_renumbered():
    from social_navigation_pyenvs_b200.large import LargeCrowd
    crowd = LargeCrowd.__new__(LargeCrowd)
    crowd._sharded_slice = True
    with pytest.raises(ValueError, match="shard"):
        crowd.renumber()
