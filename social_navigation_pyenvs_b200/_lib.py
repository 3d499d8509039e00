"""ctypes binding of libsnp_b200.so (the C ABI declared in include/snp_b200.h).

There is NO fallback: if the CUDA library is missing or does not load, importing this module's `lib()` raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SNP_B200_LIB", os.path.join(_HERE, "libsnp_b200.so"))  # override: tuning experiments only

SNP_F32, SNP_F64 = 0, 1
# bits of snp_step_opts.reserved (include/snp_b200.h)
SNP_OPT_FULL_PAIR_LOOP, SNP_OPT_NO_CULLING, SNP_OPT_MAP_WARP, SNP_OPT_MAP_BLOCK, SNP_OPT_STAGED_COPIES = 1, 2, 4, 8, 16
SNP_OPT_UNIT_SCRATCH = 32
SNP_RESET_FORCE_CTA = 1  # snp_reset_args.reserved bit 0
# field order of the SoA buffers (include/snp_b200.h)
DYN_PX, DYN_PY, DYN_VX, DYN_VY, DYN_TH, DYN_BVX, DYN_BVY, DYN_OM, DYN_DFX, DYN_DFY, DYN_FIELDS = range(11)
STAT_R, STAT_M, STAT_VD, STAT_SAFETY, STAT_FIELDS = range(5)
(ROBOT_PX, ROBOT_PY, ROBOT_VX, ROBOT_VY, ROBOT_R, ROBOT_SAFETY, ROBOT_GX, ROBOT_GY, ROBOT_TH, ROBOT_BVX, ROBOT_BVY, ROBOT_OM, ROBOT_M,
 ROBOT_VD, ROBOT_DFX, ROBOT_DFY, ROBOT_GX2, ROBOT_GY2, ROBOT_GCNT, ROBOT_SPARE, ROBOT_FIELDS) = range(21)
FLAG_COLLISION, FLAG_REACHING_GOAL, FLAG_TERMINATED, FLAG_TRUNCATED = 1, 2, 4, 8
FLAG_INFO_SHIFT = 4
FLAG_ACTUAL_COLLISION, FLAG_ACTUAL_GOAL, FLAG_TOUCHED = 1 << 7, 1 << 8, 1 << 9

c_void_p, c_int32, c_int64, c_double = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_double


class SnpCrowd(ctypes.Structure):
    _fields_ = [("E", c_int32), ("N", c_int32), ("G", c_int32), ("dtype", c_int32),
                ("dyn", c_void_p), ("stat", c_void_p), ("goals", c_void_p), ("goal_idx", c_void_p), ("goal_cnt", c_void_p),
                ("agent_params", c_void_p), ("params", c_double * 20), ("robot", c_void_p), ("walls", c_void_p),
                ("W", c_int32), ("S", c_int32), ("walls_per_env", c_int32)]


class SnpStepOpts(ctypes.Structure):
    _fields_ = [("type", c_int32), ("consider_robot", c_int32), ("symmetric", c_int32), ("numba_compat", c_int32),
                ("n_substeps", c_int32), ("robot_mode", c_int32), ("dt", c_double), ("action", c_void_p),
                ("pre_checks", c_int32), ("post_checks", c_int32), ("track_touch", c_int32), ("reserved", c_int32),
                ("consts", c_double * 6), ("time_now", c_void_p), ("flags", c_void_p), ("checks", c_void_p),
                ("respawn_bounds", c_double * 2), ("respawn", c_int32), ("robot_type", c_int32), ("robot_params", c_double * 20),
                ("dyn_out", c_void_p), ("respawn_envs", c_void_p), ("goal_idx_out", c_void_p),
                ("robot_every", c_int32), ("robot_phase", c_int32)]


class SnpLaserArgs(ctypes.Structure):
    _fields_ = [("E", c_int32), ("N", c_int32), ("dtype", c_int32), ("samples", c_int32),
                ("px", c_void_p), ("py", c_void_p), ("radius", c_void_p), ("walls", c_void_p),
                ("W", c_int32), ("S", c_int32), ("walls_per_env", c_int32), ("reserved", c_int32),
                ("pose", c_void_p), ("range", c_double), ("max_distance", c_double), ("robot_radius", c_double),
                ("ranges", c_void_p), ("hits", c_void_p), ("uncertainty", c_double), ("noise_seed", ctypes.c_uint64), ("noise_scan", ctypes.c_uint64)]


class SnpLookaheadArgs(ctypes.Structure):
    _fields_ = [("type", c_int32), ("A", c_int32), ("theta_and_omega_visible", c_int32), ("reserved", c_int32),
                ("next", c_void_p), ("actions", c_void_p), ("dt", c_double), ("rotated", c_void_p), ("rewards", c_void_p)]


class SnpValueArgs(ctypes.Structure):
    _fields_ = [("type", c_int32), ("A", c_int32), ("theta_and_omega_visible", c_int32), ("reserved", c_int32),
                ("next", c_void_p), ("actions", c_void_p), ("dt", c_double), ("gamma", c_double), ("layers", c_int32),
                ("widths", c_int32 * 7), ("weights", c_void_p), ("values", c_void_p), ("best", c_void_p), ("reached", c_void_p)]


class SnpResetArgs(ctypes.Structure):
    _fields_ = [("scenario", c_int32), ("randomize_attributes", c_int32), ("seeds", c_void_p), ("seed0", ctypes.c_uint32),
                ("reserved", ctypes.c_uint32), ("mask", c_void_p), ("circle_radius", c_double), ("robot_radius", c_double),
                ("traffic_length", c_double), ("traffic_height", c_double), ("human_mass", c_double), ("robot_mass", c_double),
                ("robot_desired_speed", c_double), ("time_now", c_void_p), ("flags", c_void_p), ("scenario_out", c_void_p),
                ("draws_out", c_void_p)]


RESET_SCENARIOS = {"circle_crossing": 0, "circular_crossing": 0, "parallel_traffic": 1, "circular_crossing_with_static_obstacles": 2,
                   "ccso_synthetic": 3, "hybrid_scenario": 4}

# every symbol include/snp_b200.h declares, with its ctypes signature
_SIGNATURES = {
    "snp_abi_version": (ctypes.c_int, []),
    "snp_last_error": (ctypes.c_char_p, []),
    "snp_device_info": (ctypes.c_int, [ctypes.POINTER(c_int32)]),
    "snp_step": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), ctypes.POINTER(SnpStepOpts), c_void_p]),
    "snp_gym_step_host": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), ctypes.POINTER(SnpStepOpts), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "snp_checks": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), ctypes.POINTER(SnpStepOpts), c_void_p]),
    "snp_laser": (ctypes.c_int, [ctypes.POINTER(SnpLaserArgs), c_void_p]),
    "snp_lookahead": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), ctypes.POINTER(SnpLookaheadArgs), c_void_p]),
    "snp_value_lookahead": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), ctypes.POINTER(SnpValueArgs), c_void_p]),
    "snp_constant_velocity": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), c_double, c_void_p, c_void_p]),
    "snp_reset": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), ctypes.POINTER(SnpResetArgs), c_void_p]),
    "snp_robot_push_out": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), c_void_p]),
    "snp_unpack_states": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), c_void_p, c_int32, c_void_p, c_void_p]),
    "snp_pack_states": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), c_void_p, c_int32, c_void_p]),
    "snp_unpack_goals": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), c_void_p, c_void_p, c_void_p]),
    "snp_rotate_goal_rows": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), c_void_p, c_void_p]),
    "snp_large_scratch_bytes": (c_int64, [c_int64, c_int64, c_int32]),
    "snp_large_scratch_bytes_units": (c_int64, [c_int64, c_int64, c_int32, c_int64]),
    "snp_large_checks": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), ctypes.POINTER(SnpStepOpts), c_void_p, c_void_p, c_int64, c_void_p]),
    "snp_large_publish": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), c_int32, c_void_p, c_int64, c_int64, c_void_p]),
    "snp_large_run_p2p": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), ctypes.POINTER(SnpStepOpts), c_void_p, c_void_p, c_int32, c_int64, c_int64, c_int32,
                                         c_int32, c_void_p, ctypes.c_uint64, c_int32, c_void_p, c_void_p, c_int64, c_void_p]),
    "snp_large_batch_scratch_bytes": (c_int64, [c_int32, c_int32, c_int32]),
    "snp_large_batch_scratch_bytes_units": (c_int64, [c_int32, c_int32, c_int32, c_int64]),
    "snp_large_batch_step": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), ctypes.POINTER(SnpStepOpts), c_void_p, c_int64, c_void_p]),
    "snp_large_tile_boxes": (ctypes.c_int, [c_void_p, c_int64, c_int32, c_void_p]),
    "snp_spatial_order_scratch_bytes": (c_int64, [c_int32, c_int32]),
    "snp_spatial_order": (ctypes.c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "snp_gather_crowd": (ctypes.c_int, [ctypes.POINTER(SnpCrowd), ctypes.POINTER(SnpCrowd), c_void_p, c_int64, c_void_p, c_void_p]),
    "snp_update_humans_parallel_host":(ctypes.c_int, [c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_int32,
                                                       c_void_p, c_double, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32,
                                                       c_void_p, c_void_p]),
    "snp_laser_host": (ctypes.c_int, [c_int32, c_int32, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_double, c_int32, c_double,
                                      c_double, c_int32, c_void_p, c_void_p]),
    "snp_measure_pipe_peak": (ctypes.c_int, [c_int32, ctypes.POINTER(c_double)]),
    "snp_debug_exp": (ctypes.c_int, [c_void_p, c_void_p, c_int32, c_void_p]),
    "snp_debug_math": (ctypes.c_int, [c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "snp_launch_count": (c_int64, [c_int32]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


class SnpError(RuntimeError):
    pass


def lib():
    """Load libsnp_b200.so (once).  Raises ImportError if it was not built -- there is no CPU fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} not found: build it with `python -m social_navigation_pyenvs_b200.build` "
                              "(the engine has no CPU or PyTorch fallback)")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the library does not export a declared symbol
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check_size(n: int) -> int:
    """A byte count from a *_scratch_bytes* function, or the ValueError of its -1."""
    if n < 0:
        raise ValueError(lib().snp_last_error().decode())
    return n


def check(rc: int):
    """Translate a negative snp_status into the exception the reference would have raised."""
    if rc == 0:
        return
    msg = lib().snp_last_error().decode()
    if rc == -1:
        raise ValueError(msg)  # forces_parallel.py:211 raises ValueError for a bad type
    if rc == -3:
        raise NotImplementedError(msg)
    raise SnpError(msg)
