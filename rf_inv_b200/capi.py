"""ctypes binding of ``librfinv_b200.so`` (the C-ABI declared in include/rfinv_b200.h).

This is the Python stand-in for the Fortran ``bind(C)`` interface block a maintainer of the reference
would add (INTEGRATION.md).  There is no CPU fallback: if the CUDA library is missing or no device is
visible every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

from .config import RfinvConfigC

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "librfinv_b200.so")

dp = C.POINTER(C.c_double)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)
u8p = C.POINTER(C.c_uint8)
i8p = C.POINTER(C.c_int8)

RFINV_OK, RFINV_ERR_ARG, RFINV_ERR_CUDA, RFINV_ERR_IO, RFINV_ERR_STATE = 0, 1, 2, 3, 4

# name -> (restype, argtypes); every symbol include/rfinv_b200.h declares
SIGNATURES = {
    "rfinv_abi_version": (C.c_int32, []),
    "rfinv_last_error": (C.c_char_p, []),
    "rfinv_device_count": (C.c_int32, []),
    "rfinv_create": (C.c_int32, [C.POINTER(RfinvConfigC), C.c_int32, C.POINTER(C.c_void_p)]),
    "rfinv_destroy": (None, [C.c_void_p]),
    "rfinv_set_stream": (C.c_int32, [C.c_void_p, C.c_uint64]),
    "rfinv_eval_batch": (C.c_int32, [C.c_void_p, C.c_int32, i32p, dp, dp, dp, dp, dp, dp, u8p]),
    "rfinv_eval_batch_flags": (C.c_int32, [C.c_void_p, C.c_int32, u8p, i32p, dp, dp, dp, dp, dp, dp, u8p]),
    "rfinv_eval_batch_begin": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, i32p, dp, dp, dp, dp, dp, u8p]),
    "rfinv_eval_batch_end": (C.c_int32, [C.c_void_p, C.c_int32]),
    "rfinv_eval_batch_device": (C.c_int32, [C.c_void_p, C.c_int32] + [C.c_uint64] * 8),
    "rfinv_format_model_batch": (C.c_int32, [C.c_void_p, C.c_int32, i32p, dp, dp, dp, i32p, dp, dp, dp, dp, u8p]),
    "rfinv_filter_traces": (C.c_int32, [C.c_void_p, C.c_int32, i32p, dp, dp]),
    "rfinv_get_r_inv": (C.c_int32, [C.c_void_p, dp]),
    "rfinv_synchronize": (C.c_int32, [C.c_void_p]),
    "rfinv_last_launch_count": (C.c_int32, [C.c_void_p]),
    "rfinv_set_timing": (C.c_int32, [C.c_void_p, C.c_int32]),
    "rfinv_get_timing": (C.c_int32, [C.c_void_p, dp]),
    "rfinv_get_quadform_form": (C.c_int32, [C.c_void_p, i32p, i32p, i32p]),
    "rfinv_measure_fp64_peak": (C.c_int32, [C.c_int32, dp, dp]),
    "rfinv_pt_init": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32]),
    "rfinv_pt_draw": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, dp]),
    "rfinv_pt_ntype": (C.c_int32, [C.c_void_p]),
    "rfinv_pt_set_logging": (C.c_int32, [C.c_void_p, C.c_int32]),
    "rfinv_pt_run": (C.c_int32, [C.c_void_p, C.c_int32]),
    "rfinv_comm_id_bytes": (C.c_int32, []),
    "rfinv_comm_create_id": (C.c_int32, [C.c_void_p]),
    "rfinv_comm_init": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    "rfinv_comm_destroy": (C.c_int32, [C.c_void_p]),
    "rfinv_comm_info": (C.c_int32, [C.c_void_p, i32p, i32p, i32p]),
    "rfinv_pt_exchange_mode": (C.c_int32, [C.c_void_p]),
    "rfinv_pt_run_distributed": (C.c_int32, [C.c_void_p, C.c_int32]),
    "rfinv_pt_reduce_outputs": (C.c_int32, [C.c_void_p]),
    "rfinv_pt_local_step": (C.c_int32, [C.c_void_p]),
    "rfinv_pt_swap_table": (C.c_int32, [C.c_void_p, C.POINTER(C.c_uint64), i32p]),
    "rfinv_pt_apply_swap": (C.c_int32, [C.c_void_p, C.c_uint64, C.c_int32]),
    "rfinv_pt_get_state": (C.c_int32, [C.c_void_p, i32p, dp, dp, dp, dp, dp, dp]),
    "rfinv_pt_get_counters": (C.c_int32, [C.c_void_p, i64p, i64p, dp, C.c_int32, i64p]),
    "rfinv_pt_iterations_done": (C.c_int32, [C.c_void_p]),
    "rfinv_pt_get_log": (C.c_int32, [C.c_void_p, i8p, i8p, i32p, i32p]),
    "rfinv_pt_get_hist": (C.c_int32, [C.c_void_p, i64p, i64p, i64p, i64p, i64p, i64p, i64p, i64p, dp, dp, dp]),
    "rfinv_pt_get_models": (C.c_int32, [C.c_void_p, C.c_int64, dp, dp, i64p]),
    "rfinv_pt_save": (C.c_int32, [C.c_void_p, C.c_char_p]),
    "rfinv_pt_restore": (C.c_int32, [C.c_void_p, C.c_char_p]),
    "rfinv_pt_group_create": (C.c_int32, [C.POINTER(C.c_void_p), C.c_int32, C.POINTER(C.c_void_p)]),
    "rfinv_pt_group_run": (C.c_int32, [C.c_void_p, C.c_int32]),
    "rfinv_pt_group_destroy": (None, [C.c_void_p]),
    "rfinv_pt_set_rank_swaps": (C.c_int32, [C.c_void_p, C.c_int32]),
    "rfinv_pt_get_rank_swaps": (C.c_int32, [C.c_void_p, i32p, i64p, i64p]),
    "rfinv_pt_set_ladder_tuning": (C.c_int32, [C.c_void_p, C.c_int32]),
    "rfinv_pt_get_ladder_tuning": (C.c_int32, [C.c_void_p, i32p, i32p]),
    "rfinv_pt_set_step_tuning": (C.c_int32, [C.c_void_p, C.c_int32, C.c_double]),
    "rfinv_pt_get_step_tuning": (C.c_int32, [C.c_void_p, i32p, C.POINTER(C.c_double), i32p, C.POINTER(C.c_double), i64p, i64p]),
    "rfinv_problem_load": (C.c_int32, [C.c_char_p, C.c_char_p, C.POINTER(C.c_void_p)]),
    "rfinv_problem_free": (None, [C.c_void_p]),
    "rfinv_problem_config": (C.POINTER(RfinvConfigC), [C.c_void_p]),
    "rfinv_problem_out_dir": (C.c_char_p, [C.c_void_p]),
    "rfinv_problem_t_end": (C.c_double, [C.c_void_p]),
    "rfinv_problem_write_copies": (C.c_int32, [C.c_void_p, C.c_char_p, C.c_char_p]),
    "rfinv_write_outputs": (C.c_int32, [C.POINTER(RfinvConfigC), C.c_char_p, C.c_int32, C.c_int64, i64p, i64p, i64p, i64p, i64p,
                                        i64p, i64p, dp, dp, dp, dp, C.c_int32, dp, dp, C.c_int64]),
}

_lib = None


class RfinvError(RuntimeError):
    def __init__(self, status: int, msg: str):
        super().__init__(f"rfinv status {status}: {msg}")
        self.status = status


def load(path: Optional[str] = None):
    """Loads the CUDA library.  Raises if it has not been built: there is no other compute path."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or SO_PATH
    if not os.path.exists(p):
        raise FileNotFoundError(
            f"{p} not found: build it with `python -m rf_inv_b200.build` (nvcc, sm_100a). "
            "rf_inv_b200 has no CPU implementation of the forward/likelihood path.")
    lib = C.CDLL(p)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def check(status: int) -> None:
    if status != RFINV_OK:
        msg = load().rfinv_last_error()
        raise RfinvError(status, msg.decode() if msg else "")
