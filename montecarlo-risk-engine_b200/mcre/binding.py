"""ctypes binding of libmcre_b200.so (include/mcre.h).

The library is the product: if it is missing or fails to load, everything that
simulates raises.  There is deliberately no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# MCRE_LIB_PATH: kernel-tuning variants of the same library (tools/tune_irc.py); never a fallback
LIB_PATH = os.environ.get("MCRE_LIB_PATH") or os.path.join(_PKG, "libmcre_b200.so")

c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int32)


class McreError(RuntimeError):
    pass


class Rng(C.Structure):
    _fields_ = [("mode", C.c_int32), ("seed", C.c_uint64), ("stream", C.c_uint64),
                ("d_z", C.c_void_p), ("d_u", C.c_void_p), ("n_paths_total", C.c_int64)]


class Shard(C.Structure):
    _fields_ = [("path_begin", C.c_int64), ("n_paths", C.c_int64), ("chunk_paths", C.c_int32)]


class IrcDesc(C.Structure):
    _fields_ = [
        ("nt", C.c_int32), ("scheme", C.c_int32), ("has_cir", C.c_int32), ("cir_deterministic", C.c_int32),
        ("vas_noise", C.c_int32), ("cir_noise", C.c_int32),
        ("vas", c_dp), ("cir", c_dp), ("cir_init", c_dp), ("chol", c_dp),
        ("n_sub", C.c_int32), ("n_dates", C.c_int32), ("n_pre_dates", C.c_int32),
        ("step_dt", c_dp), ("step_date", c_ip), ("step_vas", c_dp), ("step_cir", c_dp),
        ("date_flags", c_ip), ("date_expo", c_ip), ("date_metric", c_ip), ("date_reg", c_ip),
        ("date_float_off", c_ip), ("float_coef", c_dp), ("float_inv_tau", c_dp),
        ("n_sets", C.c_int32), ("n_expo", C.c_int32), ("n_metric", C.c_int32), ("acc_flags", C.c_int32),
        ("set_fix", c_dp), ("set_float", c_dp), ("set_threshold", c_dp), ("set_flags", c_ip), ("set_lag", c_ip),
        ("expo_coef", c_dp), ("expo_basis", c_dp), ("cva_coef", c_dp), ("lgd", C.c_double),
        ("n_units", C.c_int32), ("n_reg", C.c_int32),
        ("unit_fix", c_dp), ("unit_float", c_dp), ("unit_last_reg", c_ip), ("reg_basis", c_dp),
        ("n_berm", C.c_int32), ("berm_set", c_ip), ("berm_strike", c_dp), ("berm_sign", c_dp),
        ("date_ex_off", c_ip), ("ex_unit", c_ip), ("ex_last", c_ip), ("ex_term_off", c_ip),
        ("ex_const", c_dp), ("term_coef", c_dp), ("term_w", c_dp), ("ex_basis", c_dp),
        ("ext_numeraire", C.c_int32), ("ext_rate", C.c_double), ("ext_slot", C.c_int32),
    ]


class StorageDesc(C.Structure):
    _fields_ = [("n_sub", C.c_int32), ("n_dates", C.c_int32), ("n_pre_dates", C.c_int32), ("n_states", C.c_int32),
                ("n_basis", C.c_int32), ("log_spot0", C.c_double), ("step", c_dp), ("step_date", c_ip),
                ("date_rec", c_dp), ("numeraire", c_dp), ("noise_dim", C.c_int32), ("n_tan", C.c_int32),
                ("step_tan", c_dp), ("dlog_num", c_dp), ("n_expo", C.c_int32), ("n_pre_expo", C.c_int32),
                ("step_expo", c_ip), ("expo_numeraire", c_dp)]


RNG_PHILOX, RNG_INJECT = 0, 1
SCHEME_EULER, SCHEME_ANALYTICAL, SCHEME_QE = 0, 2, 3
DATE_HAS_CASHFLOW, DATE_HAS_EXPOSURE, DATE_HAS_METRIC, DATE_HAS_REGRESSION, DATE_HAS_EXERCISE = 1, 2, 4, 8, 16
ACC_PV, ACC_POS, ACC_NEG, ACC_CVA, ACC_SPILL = 1, 2, 4, 8, 16
IRC_MAX_SETS, IRC_MAX_UNITS, IRC_MAX_LAG, IRC_MAX_BERM = 4, 4, 4, 8

_lib = None

#: every symbol include/mcre.h declares (checked by tests/test_abi.py)
SYMBOLS = [
    "mcre_generate_paths", "mcre_correlated_normals",
    "mcre_irc_create", "mcre_irc_destroy", "mcre_irc_main_slots", "mcre_irc_presim_slots",
    "mcre_irc_presim_scratch_bytes", "mcre_irc_partial_bytes", "mcre_irc_presim", "mcre_irc_presim_tangent_slots",
    "mcre_irc_set_coefficients", "mcre_irc_solve_coefficients", "mcre_irc_set_coefficients_device", "mcre_irc_mainsim", "mcre_irc_set_pv_spill", "mcre_irc_set_path_replay", "mcre_select_locate",
    "mcre_irc_set_exercise_coefficients", "mcre_irc_lsm_scratch_bytes", "mcre_irc_lsm_forward", "mcre_lsm_step", "mcre_lsm_step_states", "mcre_lsm_step_dev", "mcre_lsm_solve_dev", "mcre_lsm_moments_batch", "mcre_lsm_step_batch", "mcre_lsm_step_tangents", "mcre_lsm_step_states_tangents",
    "mcre_lsm_prepare_equity", "mcre_lsm_prepare_equity_tangents",
    "mcre_eq_create", "mcre_eq_destroy", "mcre_eq_slots", "mcre_eq_mainsim", "mcre_eq_presim", "mcre_eq_presim_tangents", "mcre_eq_set_exposure_coef_tangents", "mcre_eq_set_exercise_exposure_coef_tangents", "mcre_eq_set_credit", "mcre_eq_set_cva_weight_spill", "mcre_eq_cva_paths", "mcre_eq_set_pv_accumulator", "mcre_eq_set_bridge_uniforms", "mcre_eq_set_exposure_accumulator", "mcre_eq_set_exposure_tangent_accumulator", "mcre_exposure_tangent_sums", "mcre_exposure_tangent_sums_paths", "mcre_eq_credit_weight_tangents", "mcre_eq_unsecured_exposures", "mcre_sum_stats",
    "mcre_storage_create", "mcre_storage_destroy", "mcre_storage_spots", "mcre_storage_backward", "mcre_storage_moment_slots", "mcre_storage_moments", "mcre_storage_solve", "mcre_storage_mainsim",
    "mcre_select_create", "mcre_select_destroy", "mcre_select_begin", "mcre_select_count",
    "mcre_select_scan", "mcre_select_compact", "mcre_select_finish",
    "mcre_tree_reduce", "mcre_dfma_peak", "mcre_fastmath_probe", "mcre_launch_count", "mcre_h2d_bytes", "mcre_last_error", "mcre_abi_version",
]


def lib():
    """Load (once) and return the CUDA library; raise loudly if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise McreError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "There is no CPU fallback for the Monte Carlo hot path.")
    L = C.CDLL(LIB_PATH)
    L.mcre_last_error.restype = C.c_char_p
    L.mcre_launch_count.restype = C.c_int64
    L.mcre_h2d_bytes.restype = C.c_int64
    L.mcre_irc_main_slots.restype = C.c_int64
    L.mcre_irc_main_slots.argtypes = [C.c_void_p]
    L.mcre_irc_presim_slots.restype = C.c_int64
    L.mcre_irc_presim_slots.argtypes = [C.c_void_p]
    L.mcre_irc_presim_scratch_bytes.restype = C.c_int64
    L.mcre_irc_presim_scratch_bytes.argtypes = [C.c_void_p, C.c_int64]
    L.mcre_irc_partial_bytes.restype = C.c_int64
    L.mcre_irc_partial_bytes.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int]
    L.mcre_irc_create.argtypes = [C.POINTER(IrcDesc), C.POINTER(C.c_void_p)]
    L.mcre_irc_destroy.argtypes = [C.c_void_p]
    L.mcre_irc_destroy.restype = None
    L.mcre_irc_presim.argtypes = [C.c_void_p, C.POINTER(Rng), C.POINTER(Shard), C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_irc_presim_tangent_slots.restype = C.c_int64
    L.mcre_irc_presim_tangent_slots.argtypes = [C.c_void_p]
    L.mcre_irc_set_coefficients.argtypes = [C.c_void_p, c_dp, C.c_void_p]
    L.mcre_irc_solve_coefficients.argtypes = [C.c_void_p, C.c_void_p, c_ip, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_irc_set_coefficients_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_irc_mainsim.argtypes = [C.c_void_p, C.POINTER(Rng), C.POINTER(Shard), C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_irc_set_pv_spill.argtypes = [C.c_void_p, C.c_void_p]
    L.mcre_irc_set_path_replay.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_select_locate.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_irc_set_exercise_coefficients.argtypes = [C.c_void_p, c_dp, c_dp, C.c_void_p]
    L.mcre_irc_lsm_scratch_bytes.restype = C.c_int64
    L.mcre_irc_lsm_scratch_bytes.argtypes = [C.c_void_p, C.c_int64]
    L.mcre_irc_lsm_forward.argtypes = [C.c_void_p, C.POINTER(Rng), C.POINTER(Shard), C.c_void_p, C.c_void_p]
    L.mcre_lsm_step.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p,
                                c_dp, C.c_double, C.c_double, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p,
                                C.c_void_p, C.c_void_p]
    L.mcre_lsm_step_states.argtypes = [C.c_int32] + list(L.mcre_lsm_step.argtypes)
    L.mcre_lsm_step_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p,
                                    C.c_void_p, C.c_void_p]
    L.mcre_lsm_solve_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_lsm_step_batch.argtypes = [C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_lsm_moments_batch.argtypes = [C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_lsm_step_tangents.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, c_dp, C.c_double,
                                         C.c_double, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p,
                                         C.c_void_p]
    L.mcre_lsm_step_states_tangents.argtypes = [C.c_int32] + list(L.mcre_lsm_step_tangents.argtypes)
    L.mcre_lsm_prepare_equity_tangents.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, c_ip, c_dp,
                                                   C.c_int32, C.c_int32, C.c_int32, c_ip, C.c_int32, C.c_double,
                                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_eq_create.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.mcre_eq_destroy.argtypes = [C.c_void_p]
    L.mcre_eq_destroy.restype = None
    L.mcre_eq_slots.argtypes = [C.c_void_p]
    L.mcre_eq_slots.restype = C.c_int64
    L.mcre_eq_mainsim.argtypes = [C.c_void_p, C.POINTER(Rng), C.POINTER(Shard), C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_eq_presim.argtypes = [C.c_void_p, C.POINTER(Rng), C.POINTER(Shard), C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]
    L.mcre_eq_presim_tangents.argtypes = [C.c_void_p, C.POINTER(Rng), C.POINTER(Shard)] + [C.c_void_p] * 7
    L.mcre_eq_set_exposure_coef_tangents.argtypes = [C.c_void_p, c_dp]
    L.mcre_eq_set_exercise_exposure_coef_tangents.argtypes = [C.c_void_p, c_dp]
    L.mcre_eq_set_credit.argtypes = [C.c_void_p, C.c_void_p]
    L.mcre_eq_set_cva_weight_spill.argtypes = [C.c_void_p, C.c_void_p]
    L.mcre_eq_cva_paths.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_void_p, C.c_void_p]
    L.mcre_eq_set_pv_accumulator.argtypes = [C.c_void_p, C.c_void_p]
    L.mcre_eq_set_bridge_uniforms.argtypes = [C.c_void_p, C.c_void_p, C.c_int32]
    L.mcre_sum_stats.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                 C.c_void_p]
    L.mcre_eq_set_exposure_accumulator.argtypes = [C.c_void_p, C.c_void_p]
    L.mcre_eq_set_exposure_tangent_accumulator.argtypes = [C.c_void_p, C.c_void_p]
    L.mcre_exposure_tangent_sums.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, c_ip, c_ip,
                                             C.c_int32, C.c_double, c_dp, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_exposure_tangent_sums_paths.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, c_ip, c_ip,
                                                   C.c_int32, C.c_double, C.c_void_p, C.c_double, C.c_void_p, C.c_int32,
                                                   C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_eq_credit_weight_tangents.argtypes = [C.c_void_p, C.c_void_p, c_dp, c_dp, C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.c_void_p]
    L.mcre_eq_unsecured_exposures.argtypes = [C.c_void_p, C.c_int64, C.c_int32, c_ip, c_ip, C.c_int32, C.c_double,
                                              C.c_void_p, C.c_void_p]
    L.mcre_tree_reduce.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]
    L.mcre_correlated_normals.argtypes = [C.POINTER(Rng), C.c_int32, C.c_int32, c_dp, C.c_int64, C.c_void_p, C.c_void_p]
    L.mcre_storage_create.argtypes = [C.POINTER(StorageDesc), C.POINTER(C.c_void_p)]
    L.mcre_storage_destroy.argtypes = [C.c_void_p]
    L.mcre_storage_destroy.restype = None
    L.mcre_storage_spots.argtypes = [C.c_void_p, C.POINTER(Rng), C.POINTER(Shard), C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_storage_backward.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    L.mcre_storage_moment_slots.argtypes = [C.c_void_p]
    L.mcre_storage_moment_slots.restype = C.c_int64
    L.mcre_storage_moments.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_int64,
                                       C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_storage_solve.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p]
    L.mcre_storage_mainsim.argtypes = [C.c_void_p, C.POINTER(Rng), C.POINTER(Shard), C.c_void_p, C.c_double, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_dfma_peak.argtypes = [c_dp, C.c_void_p]
    L.mcre_fastmath_probe.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise McreError(f"libmcre_b200 error {rc}: {lib().mcre_last_error().decode()}")


def as_dp(a):
    """numpy float64 array -> (keepalive, double*)."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(c_dp)


def as_ip(a):
    a = np.ascontiguousarray(a, dtype=np.int32)
    return a, a.ctypes.data_as(c_ip)


def launch_count():
    return int(lib().mcre_launch_count())


def h2d_bytes():
    """Bytes the library has copied host -> device so far."""
    return int(lib().mcre_h2d_bytes())
