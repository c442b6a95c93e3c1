"""Loads lib/libntm_mpc.so (the C ABI of include/ntm_mpc.h) through ctypes.

There is no CPU fallback: if the shared library is missing, or no CUDA device is usable, the
product raises -- it never routes through oracle/ or NumPy.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# NTM_MPC_LIB: another build of the same library (tools/bench_variants.py times experimental builds side by side)
LIB_PATH = os.environ.get("NTM_MPC_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "libntm_mpc.so")

NPARAM = 16
MAX_HORIZON = 128
LAYOUT_MATLAB, LAYOUT_SOA = 0, 1
PROFILE_RHO1_SQ, PROFILE_GAMMA_I, PROFILE_F_XK, PROFILE_PLANT_C, PROFILE_INNER_FIXED, PROFILE_DENSE_G = 1, 2, 4, 8, 16, 32
PROFILE_PLANT_RK4 = 64
PROFILE_TAUE_W = 128
PROFILE_LITERAL = 0
STATE_ROWS_OFF, STATE_ROWS_REFRESH, STATE_ROWS_FROZEN = 0, 1, 2
PROFILE_CONSISTENT = PROFILE_GAMMA_I | PROFILE_F_XK | PROFILE_PLANT_C

_dp = ctypes.c_void_p      # double* / int* are passed as raw addresses (host or device)
_i = ctypes.c_int
_h = ctypes.c_void_p

# every symbol include/ntm_mpc.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "ntm_create": (_i, [ctypes.POINTER(_h), _i]),
    "ntm_destroy": (_i, [_h]),
    "ntm_set_stream": (_i, [_h, ctypes.c_void_p]),
    "ntm_reset_stream": (_i, [_h]),
    "ntm_sync": (_i, [_h]),
    "ntm_last_error": (ctypes.c_char_p, []),
    "ntm_version": (_i, []),
    "ntm_device_info": (_i, [_h, ctypes.POINTER(_i), ctypes.POINTER(_i), ctypes.POINTER(_i)]),
    "ntm_launch_count": (ctypes.c_longlong, [_h]),
    "ntm_fp64_peak": (_i, [_h, _i, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]),
    "ntm_dmma_peak": (_i, [_h, _i, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]),
    "ntm_mc_stats_ub_dev": (_i, [_h, _i, _i, _i, _dp, _dp, _dp, _dp, _dp, _dp, _i, _dp, ctypes.c_double, ctypes.c_double, _dp]),
    "ntm_device_count": (_i, [ctypes.POINTER(_i)]),
    "ntm_pool_launch_count": (ctypes.c_longlong, [_i]),
    "ntm_mpc_closed_loop_multi": (_i, [_i, _dp, _i, _i, _i, _i, _i, _i, ctypes.c_double, _dp, _dp, _i, _i, _dp,
                                       _dp, _dp, _dp, _dp, _dp, _dp, _dp]),
    "ntm_mpc_closed_loop_rec_dev": (_i, [_h, _i, _i, _i, _i, _i, ctypes.c_double, _dp, _dp, _i, _i, _dp, _dp, _dp, _dp]),
}


def rec_doubles(k_sim: int) -> int:
    """NTM_REC_DOUBLES(k_sim): doubles per scenario of the packed record [xk | uk | cost | status]."""
    return 3 * k_sim + 4


def kf_doubles() -> int:
    """NTM_KF_DOUBLES: doubles per scenario of an observer record (``ntm_kf_step``): xhat, p11, p21, p22, steps."""
    return 6


def ctrl_doubles(N: int) -> int:
    """NTM_CTRL_DOUBLES(N): doubles per scenario of a controller record (``ntm_mpc_step``)."""
    return 7 * N + 7


for _sfx in ("", "_dev"):
    SYMBOLS["ntm_rho" + _sfx] = (_i, [_h, _i, _i, _i, _dp, _dp, _i, _dp, _dp, _dp])
    SYMBOLS["ntm_lpv_AB" + _sfx] = (_i, [_h, _i, _i, _dp, _dp, _dp, _dp, _i, _dp, _dp])
    SYMBOLS["ntm_condense" + _sfx] = (_i, [_h, _i, _i, _i, _i, _dp, _dp, _dp, _dp, _i, _dp, _dp, _dp])
    SYMBOLS["ntm_hessian_grad" + _sfx] = (_i, [_h, _i, _i, _i, _dp, _dp, _dp, _dp, _dp, _i, _dp, _dp])
    SYMBOLS["ntm_qp_box" + _sfx] = (_i, [_h, _i, _i, _i, _dp, _dp, _dp, _dp, _i, _dp, _dp, _dp])
    SYMBOLS["ntm_qp_ineq" + _sfx] = (_i, [_h, _i, _i, _i, _i, _dp, _dp, _dp, _dp, _i, _dp, _dp, _dp, _dp, _dp])
    SYMBOLS["ntm_mc_stats" + _sfx] = (_i, [_h, _i, _i, _i, _dp, _dp, _dp, _dp, _dp, _i, _dp, ctypes.c_double,
                                            ctypes.c_double, _dp])
    SYMBOLS["ntm_getWLc" + _sfx] = (_i, [_h, _i, _i, _i, _dp, _dp, _dp, _dp, _dp, _dp, _dp])
    SYMBOLS["ntm_plant_step" + _sfx] = (_i, [_h, _i, _i, _i, _dp, _dp, _dp, _i, _dp])
    SYMBOLS["ntm_mpc_closed_loop" + _sfx] = (_i, [_h, _i, _i, _i, _i, _i, _i, ctypes.c_double, _dp, _dp, _i,
                                                  _dp, _dp, _dp, _dp, _dp, _dp, _dp])
    SYMBOLS["ntm_mpc_step" + _sfx] = (_i, [_h, _i, _i, _i, _i, _i, ctypes.c_double, _dp, _dp, _i, _dp, _dp, _dp, _dp,
                                           _dp, _dp])
    SYMBOLS["ntm_mpc_step_sc" + _sfx] = (_i, [_h, _i, _i, _i, _i, _i, ctypes.c_double, _dp, _dp, _i, _i, _dp, _dp, _dp,
                                              _dp, _dp, _dp, _dp])
    SYMBOLS["ntm_mpc_closed_loop_perturbed" + _sfx] = (_i, [_h, _i, _i, _i, _i, _i, _i, ctypes.c_double, _dp, _dp, _i,
                                                            _dp, _i, _i, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp])
    SYMBOLS["ntm_mpc_closed_loop_perturbed_sc" + _sfx] = (_i, [_h, _i, _i, _i, _i, _i, _i, ctypes.c_double, _dp, _dp,
                                                               _i, _i, _dp, _dp, _i, _i, _dp, _dp, _dp, _dp, _dp, _dp,
                                                               _dp, _dp, _dp])
    SYMBOLS["ntm_kf_step" + _sfx] = (_i, [_h, _i, _i, _i, _dp, _dp, _dp, _i, _dp, _dp, _dp])
    SYMBOLS["ntm_mpc_closed_loop_observed" + _sfx] = (_i, [_h, _i, _i, _i, _i, _i, _i, ctypes.c_double, _dp, _dp, _i,
                                                           _i, _dp, _dp, _i, _i, _dp, _dp, _dp, _dp, _dp, _dp, _dp,
                                                           _dp, _dp, _dp, _dp])
    SYMBOLS["ntm_mpc_closed_loop_sc" + _sfx] = (_i, [_h, _i, _i, _i, _i, _i, _i, ctypes.c_double, _dp, _dp, _i, _i, _dp,
                                                     _dp, _dp, _dp, _dp, _dp, _dp, _dp])

_lib = None


class NtmError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NtmError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  There is no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        lenient = bool(os.environ.get("NTM_MPC_LIB"))   # an older experimental build may lack the newest entry points
        for name, (res, args) in SYMBOLS.items():
            if lenient and not hasattr(lib, name):
                continue
            fn = getattr(lib, name)          # AttributeError here = header and library out of sync
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().ntm_last_error().decode("utf-8", "replace")
        raise NtmError(f"libntm_mpc error {rc}: {msg}")
