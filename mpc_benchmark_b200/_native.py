"""ctypes binding of libmpcb200.so (include/mpcb200.h).  There is no CPU fallback: importing works without a
GPU (so the ABI can be inspected), but every compute entry point raises if the library or CUDA is missing."""
import ctypes as C
import os

import numpy as np

from . import _abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MPCB200_LIB", os.path.join(_HERE, "libmpcb200.so"))  # override only for profiling builds
_lib = None
dp = C.POINTER(C.c_double)

EXPORTS = [
    "mpc_create", "mpc_destroy", "mpc_last_error", "mpc_setup", "mpc_update_knots", "mpc_update_terms", "mpc_cycle", "mpc_set_x0", "mpc_shift_multipliers", "mpc_reconfigure",
    "mpc_run", "mpc_run_pipelined", "mpc_run_device", "mpc_tick", "mpc_get_results", "mpc_export_results_device", "mpc_result_ptrs", "mpc_get_stage_data", "mpc_last_launches", "mpc_last_device_ms",
    "mpc_get_feedback", "mpc_last_kernel_ms", "mpc_last_kernel_launches", "mpc_set_profiling",
    "mpc_qp_create", "mpc_qp_destroy", "mpc_qp_last_error", "mpc_qp_default_settings", "mpc_qp_update", "mpc_qp_solve", "mpc_qp_solve_device",
    "mpc_qp_last_device_ms", "mpc_qp_abi_sizeof", "mpc_qp_assemble_id", "mpc_qp_debug_phases", "mpc_qp_assemble_id_from_state", "mpc_rbd_terms", "mpc_rbd_terms_device",
    "mpc_ikid_terms", "mpc_ikid_terms_device", "mpc_qp_assemble_ikid_from_state", "mpc_gait_setup", "mpc_gait_tick", "mpc_get_knots", "mpc_set_tail_warmstart",
    "mpc_reset_multipliers", "mpc_debug_lq", "mpc_debug_gemm_tn", "mpc_debug_phases", "mpc_workspace_bytes", "mpc_abi_sizeof", "mpc_measure_fp64_peak", "mpc_measure_fp64_peak_dmma",
]


class NativeError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` (no CPU fallback exists)")
        L = C.CDLL(LIB_PATH)
        L.mpc_create.restype = C.c_void_p
        L.mpc_create.argtypes = [C.POINTER(_abi.Robot), C.POINTER(_abi.Config), C.c_int32, C.c_int32]
        L.mpc_destroy.argtypes = [C.c_void_p]
        L.mpc_last_error.restype = C.c_char_p
        L.mpc_setup.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, dp]
        L.mpc_update_knots.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]
        L.mpc_update_terms.argtypes = [C.c_void_p, C.c_void_p]
        L.mpc_cycle.argtypes = [C.c_void_p, C.c_void_p]
        L.mpc_set_x0.argtypes = [C.c_void_p, dp]
        L.mpc_shift_multipliers.argtypes = [C.c_void_p, C.c_int32]
        L.mpc_reconfigure.argtypes = [C.c_void_p, C.POINTER(_abi.Robot), C.POINTER(_abi.Config)]
        L.mpc_run.argtypes = [C.c_void_p, dp, dp, C.c_int32]
        L.mpc_run_pipelined.argtypes = [C.c_void_p, dp, dp, C.c_int32, C.c_int32, dp, dp, dp, C.c_void_p]
        L.mpc_tick.argtypes = [C.c_void_p, C.c_void_p, dp, C.c_int32, C.c_int32]
        L.mpc_run_device.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_int32, C.c_uint64]
        L.mpc_get_results.argtypes = [C.c_void_p, dp, dp, dp, dp, dp, C.c_void_p]
        L.mpc_export_results_device.argtypes = [C.c_void_p] + [C.c_uint64] * 5
        L.mpc_result_ptrs.argtypes = [C.c_void_p] + [C.POINTER(C.c_uint64)] * 4
        L.mpc_get_stage_data.argtypes = [C.c_void_p, C.c_int32, dp, dp]
        L.mpc_last_launches.argtypes = [C.c_void_p]
        L.mpc_last_device_ms.argtypes = [C.c_void_p]
        L.mpc_last_device_ms.restype = C.c_double
        L.mpc_get_feedback.argtypes = [C.c_void_p, C.c_int32, dp]
        L.mpc_last_kernel_ms.argtypes = [C.c_void_p, C.c_int32]
        L.mpc_last_kernel_ms.restype = C.c_double
        L.mpc_last_kernel_launches.argtypes = [C.c_void_p, C.c_int32]
        L.mpc_set_profiling.argtypes = [C.c_void_p, C.c_int32]
        L.mpc_debug_lq.argtypes = [C.c_void_p, dp, dp, C.c_int32] + [dp] * 6
        L.mpc_debug_gemm_tn.argtypes = [C.c_int32, C.c_int32, C.c_int32, dp, C.c_int32, dp, C.c_int32, dp, C.c_int32]
        L.mpc_debug_phases.argtypes = [C.c_void_p, dp]
        L.mpc_reset_multipliers.argtypes = [C.c_void_p, C.c_uint64]
        L.mpc_workspace_bytes.argtypes = [C.c_void_p]
        L.mpc_workspace_bytes.restype = C.c_uint64
        L.mpc_abi_sizeof.argtypes = [C.c_int32]
        L.mpc_measure_fp64_peak.argtypes = [C.c_int32]
        L.mpc_measure_fp64_peak.restype = C.c_double
        L.mpc_measure_fp64_peak_dmma.argtypes = [C.c_int32]
        L.mpc_measure_fp64_peak_dmma.restype = C.c_double
        # include/mpcqp_b200.h (batched dense QP, SURVEY 8f row f-3)
        i64, u64, i32p = C.c_int64, C.c_uint64, C.POINTER(C.c_int32)
        L.mpc_qp_create.restype = C.c_void_p
        L.mpc_qp_create.argtypes = [C.c_int32] * 6
        L.mpc_qp_destroy.argtypes = [C.c_void_p]
        L.mpc_qp_last_error.restype = C.c_char_p
        L.mpc_qp_default_settings.argtypes = [C.POINTER(_abi.QPSettings)]
        L.mpc_qp_update.argtypes = [C.c_void_p, C.c_int32] + [dp, i64] * 9
        L.mpc_qp_solve.argtypes = [C.c_void_p, C.POINTER(_abi.QPSettings), dp, dp, dp, C.c_void_p]
        L.mpc_qp_solve_device.argtypes = [C.c_void_p, C.c_int32, C.POINTER(_abi.QPSettings)] + [u64, i64] * 9 + [u64] * 5
        L.mpc_qp_last_device_ms.argtypes = [C.c_void_p]
        L.mpc_qp_last_device_ms.restype = C.c_double
        L.mpc_qp_abi_sizeof.argtypes = [C.c_int32]
        L.mpc_qp_debug_phases.argtypes = [C.c_void_p, dp]
        L.mpc_qp_assemble_id_from_state.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, dp, dp, dp, i32p] + [C.c_double] * 4
        L.mpc_rbd_terms.argtypes = [C.c_void_p, C.c_int32] + [dp] * 6
        L.mpc_rbd_terms_device.argtypes = [C.c_void_p, C.c_int32] + [u64] * 7
        L.mpc_ikid_terms.argtypes = [C.c_void_p, C.c_int32, dp, i32p, dp] + [dp] * 8
        L.mpc_ikid_terms_device.argtypes = [C.c_void_p, C.c_int32, u64, i32p, dp] + [u64] * 9
        L.mpc_qp_assemble_ikid_from_state.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, dp, dp, dp, i32p, dp, dp, i32p, dp] + [C.c_double] * 3
        L.mpc_gait_setup.argtypes = [C.c_void_p, C.POINTER(_abi.Gait), i32p, dp]
        L.mpc_gait_tick.argtypes = [C.c_void_p, dp, dp]
        L.mpc_get_knots.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.mpc_set_tail_warmstart.argtypes = [C.c_void_p, C.c_int32]
        L.mpc_qp_assemble_id.argtypes = [C.c_void_p, C.c_int32] + [dp] * 6 + [i32p] + [C.c_double] * 3
        _lib = L
    return _lib


def last_error():
    return lib().mpc_last_error().decode()


def check(rc, what):
    if rc != 0:
        raise NativeError(f"{what} failed: {last_error()}")


def ptr(a):
    if a is None:
        return None
    assert isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags["C_CONTIGUOUS"], "expected contiguous float64 array"
    return a.ctypes.data_as(dp)
