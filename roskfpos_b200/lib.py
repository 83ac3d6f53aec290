"""ctypes binding of libkfpos_b200.so (the C ABI declared in include/kfpos_b200.h).

The library is built in-tree by roskfpos_b200/csrc/Makefile (see
__graft_entry__.build()).  There is no fallback: if the shared object is missing
the import of this module's `lib()` raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# KFPOS_B200_SO: another build of the same library (kernel variants under profiles/, never a different backend)
SO_PATH = os.environ.get("KFPOS_B200_SO") or os.path.join(_HERE, "csrc", "libkfpos_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "kfpos_b200.h")

MODEL_ML, MODEL_T6, MODEL_K8, MODEL_T9 = 0, 1, 2, 3
FMT_F64_M, FMT_I32_MM, FMT_U16_MM = 0, 1, 2
ST_NO_MEAS, ST_ML_FEW, ST_SINGULAR, ST_NAN, ST_ML_NAN, ST_MAXITER, ST_ASYM_R = 1, 2, 4, 8, 16, 32, 64
ST_Z_GATE = 128
ST_UNINIT = 256
HIST_ERR, HIST_ERR_XY, HIST_NEES = 0, 1, 2
SCORE_COLS = 8  # KFPOS_SCORE_COLS: the columns of kfpos_batch_score_selection
CRLB_PRESENT, CRLB_LOS, CRLB_USED = 0, 1, 2
CRLB_COLS = 4  # KFPOS_CRLB_COLS: the columns of kfpos_batch_crlb
MAX_OBSTACLES = 32  # KFPOS_MAX_OBSTACLES: the boxes of kfpos_synth_toa_ranges_geo


class KfposConfig(C.Structure):
    _fields_ = [
        ("accel_noise", C.c_double), ("jolt", C.c_double), ("initial_angle", C.c_double),
        ("ignore_worst_anchor", C.c_int32), ("ml2d_zero_tentative_z", C.c_int32),
        ("ignore_cost_threshold", C.c_double),
        ("use2d", C.c_int32), ("variant", C.c_int32), ("num_ignored_rangings", C.c_int32),
        ("best_mode", C.c_int32),
        ("min_z", C.c_double), ("max_z", C.c_double), ("ml_start", C.c_double * 3),
        ("use_fixed_height", C.c_int32), ("tag_id", C.c_int32), ("fixed_height", C.c_double),
        ("px4_use_fixed_sensor_height", C.c_int32), ("ml_exact_order", C.c_int32),
        ("px4_sensor_height", C.c_double), ("px4_arm_p0", C.c_double), ("px4_arm_p1", C.c_double),
        ("px4_sensor_init_angle", C.c_double), ("px4_cov_velocity", C.c_double),
        ("px4_cov_gyro_z", C.c_double),
        ("imu_use_fixed_cov_acc", C.c_int32), ("imu_use_fixed_cov_gyro_z", C.c_int32),
        ("imu_cov_acc", C.c_double), ("imu_cov_gyro_z", C.c_double),
        ("mag_angle_offset", C.c_double), ("mag_cov", C.c_double),
        ("ml_initial_position", C.c_int32), ("_reserved0", C.c_int32),
    ]


EV_TOA, EV_PX4, EV_IMU, EV_MAG, EV_COMPASS = 0, 1, 2, 3, 4
EV_ROWS = {EV_PX4: 5, EV_IMU: 3, EV_MAG: 2, EV_COMPASS: 1}


class KfposEvent(C.Structure):
    _fields_ = [("kind", C.c_int32), ("_pad", C.c_int32), ("dt", C.c_double), ("offset", C.c_int64),
                ("aux", C.c_double * 9)]


class KfposSynthEvent(C.Structure):
    _fields_ = [("kind", C.c_int32), ("global_index", C.c_int32), ("t", C.c_double), ("offset", C.c_int64)]


class KfposSynthToa(C.Structure):
    """kfpos_synth_toa: the ranging generator of kfpos_synth_toa_ranges."""
    _fields_ = [("seed", C.c_uint64), ("first_filter", C.c_int64), ("first_epoch", C.c_int64),
                ("tag_z", C.c_double), ("sigma_r", C.c_double), ("p_missing", C.c_double), ("p_nlos", C.c_double),
                ("nlos_mean", C.c_double)]


class KfposObstacle(C.Structure):
    """kfpos_obstacle: an axis-aligned box of kfpos_synth_toa_ranges_geo."""
    _fields_ = [("lo", C.c_double * 3), ("hi", C.c_double * 3), ("excess_per_m", C.c_double), ("spread", C.c_double),
                ("p_loss", C.c_double)]


_LIB = None

# name -> (restype, argtypes); every symbol include/kfpos_b200.h declares
_VP, _I, _I64, _D = C.c_void_p, C.c_int, C.c_int64, C.c_double
SIGNATURES = {
    "kfpos_config_default": (None, [C.POINTER(KfposConfig)]),
    "kfpos_config_load_xml": (_I, [C.POINTER(KfposConfig), C.c_char_p]),
    "kfpos_strerror": (C.c_char_p, [_I]),
    "kfpos_abi_version": (_I, []),
    "kfpos_batch_create": (_I, [C.POINTER(_VP), _I, _I, _I64, C.POINTER(KfposConfig)]),
    "kfpos_batch_destroy": (None, [_VP]),
    "kfpos_batch_size": (_I64, [_VP]),
    "kfpos_batch_state_dim": (_I, [_VP]),
    "kfpos_batch_set_anchors": (_I, [_VP, _I, _VP]),
    "kfpos_batch_set_state": (_I, [_VP, _VP, _VP, _VP]),
    "kfpos_batch_get_state": (_I, [_VP, _VP, _VP, _VP, _VP]),
    "kfpos_batch_get_latches": (_I, [_VP, _VP, _VP, _VP, _VP]),
    "kfpos_batch_set_latches": (_I, [_VP, _VP, _VP, _VP, _VP]),
    "kfpos_batch_step_toa": (_I, [_VP, _D, _VP, _I, _D, _VP, _VP]),
    "kfpos_batch_replay_toa": (_I, [_VP, _I, _VP, _VP, _I, _D, _VP, _VP, _VP, _VP]),
    "kfpos_batch_replay_epochs": (_I, [_VP, _I, _VP, _VP, _I, _D, _VP, _VP, _VP]),
    "kfpos_batch_step_px4": (_I, [_VP, _D, _VP, _VP, _VP, _VP, _VP, _VP]),
    "kfpos_batch_step_imu": (_I, [_VP, _D, _VP, _VP, _VP, _VP, _VP]),
    "kfpos_batch_step_mag": (_I, [_VP, _D, _VP, _VP]),
    "kfpos_batch_step_compass": (_I, [_VP, _D, _VP, _VP]),
    "kfpos_batch_replay_events": (_I, [_VP, _I, _VP, _VP, _I, _D, _VP, _VP, _I64, _VP, _VP]),
    "kfpos_batch_get_pose": (_I, [_VP, _D, _VP, _VP, _VP]),
    "kfpos_batch_get_pose_msg": (_I, [_VP, _D, _VP, _VP, _VP]),
    "kfpos_batch_ml_solve": (_I, [_VP, _VP, _I, _D, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "kfpos_batch_get_counters": (_I, [_VP, C.POINTER(C.c_double * 8), _I, _VP]),
    "kfpos_batch_error_stats": (_I, [_VP, _VP, C.POINTER(C.c_double * 4), _VP]),
    "kfpos_batch_set_truth": (_I, [_VP, _VP, _VP]),
    "kfpos_stats_allreduce": (_I, [_VP, _VP, _VP, C.POINTER(C.c_double * 6), _VP]),
    "kfpos_measure_fp64_peak": (_I, [_I, C.POINTER(C.c_double)]),
    "kfpos_synth_k8": (_I, [_I, _I64, _I64, C.c_uint64, _I, _VP, _D, _D, _I, _VP, _D, _I64, _I64, _VP, _VP, _VP, _VP, _VP]),
    "kfpos_selftest_math": (_I, [_I, _I64, _VP, _VP, _VP, _VP, _VP]),
    "kfpos_selftest_ieee": (_I, [_I, _I64, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "kfpos_assemble_epochs": (_I, [_I, _I64, _I64, _I, _VP, _VP, _VP, _VP, _VP, _I64, _I, _D, _VP, _VP, _VP, _VP, _VP]),
    "kfpos_assemble_epochs_t": (_I, [_I, _I64, _I64, _I, _VP, _VP, _VP, _VP, _VP, _I64, _I, _D, _VP, _VP, _VP, _VP, _VP, _VP]),
    "kfpos_merge_streams": (_I, [_I, _I64, _I, _I64, _VP, _VP, _VP, _VP, _VP, _VP, _I, _VP, _D, _VP, _VP, _VP, _VP, _VP,
                                 _VP, _VP, _VP]),
    "kfpos_batch_replay_events_ragged": (_I, [_VP, _I, _VP, _VP, _VP, _I, _D, _VP, _VP, _I64, _VP, _VP]),
    "kfpos_batch_set_truth_traj": (_I, [_VP, _I64, _VP, _VP]),
    "kfpos_batch_epoch_stats": (_I, [_VP, _I64, _VP, _VP]),
    "kfpos_epoch_stats_allreduce": (_I, [_VP, _VP, _I64, _VP, _VP]),
    "kfpos_synth_k8_truth": (_I, [_I, _I64, _I64, C.c_uint64, _I, _VP, _D, _VP, _VP]),
    "kfpos_synth_toa_ranges": (_I, [_I, _I64, _I, _VP, _I, _VP, C.POINTER(KfposSynthToa), _I, _VP, _VP]),
    "kfpos_batch_set_error_hist": (_I, [_VP, _I, _I, _VP]),
    "kfpos_batch_error_hist": (_I, [_VP, _I64, _VP, _VP]),
    "kfpos_error_hist_allreduce": (_I, [_VP, _VP, _I64, _VP, _VP]),
    "kfpos_synth_toa_ranges_nlos": (_I, [_I, _I64, _I, _VP, _I, _VP, C.POINTER(KfposSynthToa), _I, _VP, _VP, _VP]),
    "kfpos_batch_score_selection": (_I, [_VP, _I, _VP, _I, _VP, _VP, _VP, _VP]),
    "kfpos_batch_crlb": (_I, [_VP, _I, _I, _VP, _VP, _I, _D, _VP, _VP, _VP, _VP, _VP]),
    "kfpos_synth_toa_ranges_geo": (_I, [_I, _I64, _I, _VP, _I, _VP, C.POINTER(KfposSynthToa), _I, _VP, _I, _VP, _VP,
                                        _VP]),
}
ASM_FIX_ROW_CLEAR = 1


class KfposError(RuntimeError):
    def __init__(self, code: int, what: str):
        self.code = code
        super().__init__(f"{what}: {lib().kfpos_strerror(code).decode()} ({code})")


def lib():
    """Loads libkfpos_b200.so; raises if the CUDA extension was not built."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(
                f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` (nvcc, sm_100a). roskfpos_b200 has no CPU fallback.")
        l = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _LIB = l
    return _LIB


def check(code: int, what: str) -> None:
    if code != 0:
        raise KfposError(code, what)
