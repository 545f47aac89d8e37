"""ctypes binding of the C ABI declared in include/nmch_b200.h (one-to-one, no logic)."""
from __future__ import annotations

import ctypes as C
import os

from . import _build

METHOD_FE, METHOD_EM, METHOD_QE = 0, 1, 2
FLOOR_ABS, FLOOR_PLUS = 0, 1
RNG_PHILOX, RNG_XORWOW_COMPAT, RNG_PHILOX_COMPAT, RNG_MRG32K3A_COMPAT, RNG_PHILOX_DENSE, RNG_XORWOW_FAST = 0, 1, 2, 3, 4, 5

OK, ERR_ARG, ERR_CUDA, ERR_STATE, ERR_NCCL = 0, -1, -2, -3, -4


class NmchParams(C.Structure):
    _fields_ = [
        ("NTPB", C.c_int), ("NB", C.c_int),
        ("T", C.c_float), ("S_0", C.c_float), ("v_0", C.c_float), ("r", C.c_float), ("k", C.c_float),
        ("rho", C.c_float), ("theta", C.c_float), ("sigma", C.c_float),
        ("N", C.c_int), ("method", C.c_int), ("floor", C.c_int), ("rng", C.c_int), ("device", C.c_int),
        ("n_paths", C.c_ulonglong), ("first_path", C.c_ulonglong), ("n_local", C.c_ulonglong),
        ("paths_per_thread", C.c_int), ("block_threads", C.c_int),
    ]


class NmchMoments(C.Structure):
    _fields_ = [("sum_payoff", C.c_double), ("sum_payoff_sq", C.c_double), ("n_paths", C.c_ulonglong),
                ("exec_ms", C.c_float)]


class NmchStrikeMoments(C.Structure):
    _fields_ = [("strike", C.c_float), ("sum_payoff", C.c_double), ("sum_payoff_sq", C.c_double),
                ("sum_delta", C.c_double), ("sum_itm", C.c_double), ("n_paths", C.c_ulonglong), ("exec_ms", C.c_float)]


class NmchGreekMoments(C.Structure):
    _fields_ = [("strike", C.c_float), ("sum_payoff", C.c_double), ("sum_payoff_sq", C.c_double),
                ("sum_delta", C.c_double), ("sum_itm", C.c_double), ("sum_vega", C.c_double), ("sum_vega_sq", C.c_double),
                ("n_paths", C.c_ulonglong), ("exec_ms", C.c_float)]


# direction order of the sensitivity sums (NMCH_SENS_* of include/nmch_b200.h)
SENS_V0, SENS_KAPPA, SENS_THETA, SENS_SIGMA, SENS_RHO, SENS_COUNT = 0, 1, 2, 3, 4, 5
SENS_NAMES = ("v0", "kappa", "theta", "sigma", "rho")


class NmchSensitivityMoments(C.Structure):
    _fields_ = [("strike", C.c_float), ("sum_payoff", C.c_double), ("sum_payoff_sq", C.c_double),
                ("sum_delta", C.c_double), ("sum_itm", C.c_double), ("sum_sens", C.c_double * SENS_COUNT),
                ("sum_sens_sq", C.c_double * SENS_COUNT), ("n_paths", C.c_ulonglong), ("exec_ms", C.c_float)]


class NmchLaunchInfo(C.Structure):
    _fields_ = [("grid_x", C.c_int), ("grid_y", C.c_int), ("block_threads", C.c_int),
                ("paths_per_thread", C.c_int), ("regs_per_thread", C.c_int), ("sm_count", C.c_int),
                ("kernel_param_bytes", C.c_int), ("kernel_launches", C.c_ulonglong)]


EXPORTS = [
    "nmch_engine_create", "nmch_engine_init", "nmch_engine_set_params", "nmch_engine_seek", "nmch_engine_compute",
    "nmch_engine_compute_async", "nmch_engine_explore", "nmch_engine_explore_async",
    "nmch_engine_compute_paths", "nmch_engine_compute_strikes", "nmch_engine_compute_strikes_async",
    "nmch_engine_compute_greeks", "nmch_engine_compute_greeks_async", "nmch_group_compute_greeks",
    "nmch_engine_compute_sensitivities", "nmch_engine_compute_sensitivities_async", "nmch_group_compute_sensitivities",
    "nmch_engine_finalize", "nmch_engine_destroy", "nmch_engine_init_ms", "nmch_engine_check", "nmch_checked_build", "nmch_checked_selftest",
    "nmch_engine_launch_info", "nmch_group_create", "nmch_group_init", "nmch_group_set_params", "nmch_group_compute",
    "nmch_group_explore", "nmch_group_compute_strikes", "nmch_group_finalize", "nmch_group_destroy", "nmch_group_init_ms", "nmch_group_size",
    "nmch_status_string", "nmch_last_error", "nmch_device_count", "nmch_version",
]

_lib = None


class NmchError(RuntimeError):
    def __init__(self, status: int, detail: str):
        super().__init__(f"nmch_b200 status {status}: {detail}")
        self.status = status


def load() -> C.CDLL:
    """Load libnmch_b200.so; raises (never falls back) when it is missing and cannot be built."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("NMCH_B200_LIB") or _build.LIB     # override: tuning builds of the same ABI
    if path == _build.LIB and not os.path.exists(path):
        _build.build()
    L = C.CDLL(path)
    vp, f32p, f64p = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_double)
    L.nmch_engine_create.argtypes = [C.POINTER(NmchParams), C.POINTER(vp)]
    L.nmch_engine_init.argtypes = [vp, C.c_ulonglong]
    L.nmch_engine_set_params.argtypes = [vp, C.c_float, C.c_float, C.c_float]
    L.nmch_engine_seek.argtypes = [vp, C.c_ulonglong]
    L.nmch_engine_compute.argtypes = [vp, C.POINTER(NmchMoments)]
    L.nmch_engine_compute_async.argtypes = [vp, vp, vp]
    L.nmch_engine_explore.argtypes = [vp, f32p, f32p, f32p, C.c_int, C.POINTER(NmchMoments)]
    L.nmch_engine_explore_async.argtypes = [vp, vp, f32p, f32p, f32p, C.c_int, vp]
    L.nmch_engine_compute_paths.argtypes = [vp, f32p, f32p, C.c_ulonglong, C.POINTER(NmchMoments)]
    L.nmch_engine_compute_strikes.argtypes = [vp, f32p, C.c_int, C.POINTER(NmchStrikeMoments)]
    L.nmch_engine_compute_strikes_async.argtypes = [vp, vp, f32p, C.c_int, vp]
    L.nmch_group_compute_strikes.argtypes = [vp, f32p, C.c_int, C.POINTER(NmchStrikeMoments)]
    L.nmch_engine_compute_greeks.argtypes = [vp, f32p, C.c_int, C.POINTER(NmchGreekMoments)]
    L.nmch_engine_compute_greeks_async.argtypes = [vp, vp, f32p, C.c_int, vp]
    L.nmch_group_compute_greeks.argtypes = [vp, f32p, C.c_int, C.POINTER(NmchGreekMoments)]
    L.nmch_engine_compute_sensitivities.argtypes = [vp, f32p, C.c_int, C.POINTER(NmchSensitivityMoments)]
    L.nmch_engine_compute_sensitivities_async.argtypes = [vp, vp, f32p, C.c_int, vp]
    L.nmch_group_compute_sensitivities.argtypes = [vp, f32p, C.c_int, C.POINTER(NmchSensitivityMoments)]
    L.nmch_engine_check.argtypes = [vp]
    L.nmch_checked_selftest.argtypes = [vp]
    L.nmch_engine_finalize.argtypes = [vp]
    L.nmch_engine_destroy.argtypes = [vp]
    L.nmch_engine_destroy.restype = None
    L.nmch_engine_init_ms.argtypes = [vp]
    L.nmch_engine_init_ms.restype = C.c_float
    L.nmch_engine_launch_info.argtypes = [vp, C.POINTER(NmchLaunchInfo)]
    L.nmch_group_create.argtypes = [C.POINTER(NmchParams), C.c_int, C.POINTER(vp)]
    L.nmch_group_init.argtypes = [vp, C.c_ulonglong]
    L.nmch_group_set_params.argtypes = [vp, C.c_float, C.c_float, C.c_float]
    L.nmch_group_compute.argtypes = [vp, C.POINTER(NmchMoments)]
    L.nmch_group_explore.argtypes = [vp, f32p, f32p, f32p, C.c_int, C.POINTER(NmchMoments)]
    L.nmch_group_finalize.argtypes = [vp]
    L.nmch_group_destroy.argtypes = [vp]
    L.nmch_group_destroy.restype = None
    L.nmch_group_init_ms.argtypes = [vp]
    L.nmch_group_init_ms.restype = C.c_float
    L.nmch_group_size.argtypes = [vp]
    L.nmch_status_string.argtypes = [C.c_int]
    L.nmch_status_string.restype = C.c_char_p
    L.nmch_last_error.restype = C.c_char_p
    L.nmch_version.restype = C.c_char_p
    _lib = L
    return L


def check(status: int) -> None:
    if status != OK:
        L = load()
        raise NmchError(status, f"{L.nmch_status_string(status).decode()}: {L.nmch_last_error().decode()}")
