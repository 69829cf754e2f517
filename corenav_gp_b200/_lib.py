"""ctypes binding of libcngp.so (include/cngp.h).  There is no CPU fallback: a missing library is an ImportError-like
RuntimeError, and cngp_create fails without a CUDA device."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcngp.so")

MAX_OPS = 32
MAX_PARAMS = 24
MAX_N = 256
MEM_HOST, MEM_DEVICE = 0, 1
PROF_FIT, PROF_VAR, PROF_GRAD, PROF_LOOKAHEAD, PROF_LARGE, PROF_MISC = range(6)
PERWIN_P, PERWIN_Q, PERWIN_STM, PERWIN_H, PERWIN_POS = 1, 2, 4, 8, 16

c_i32, c_i64, c_dp, c_ip, c_vp = C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p


class Kernel(C.Structure):
    _fields_ = [("n_ops", c_i32), ("ops", c_i32 * MAX_OPS), ("n_params", c_i32)]


class Config(C.Structure):
    _fields_ = [("device", c_i32), ("jitter_retry", c_i32), ("scratch_bytes", c_i64), ("precision", c_i32),
                ("reserved", c_i32 * 7)]


class StopConfig(C.Structure):
    _fields_ = [("v_nom", C.c_double), ("floor_a", C.c_double), ("floor_b", C.c_double), ("track", C.c_double),
                ("scale", C.c_double), ("thresh", C.c_double), ("ratio", c_i32), ("fix_h_packing", c_i32),
                ("init_llh", C.c_double * 3), ("init_ecef", C.c_double * 3)]


class SlipConfig(C.Structure):   # cngp_slip_config
    _fields_ = [("wheel_radius", C.c_double), ("cmd_min", C.c_double), ("rear_min", C.c_double),
                ("arm_delay", C.c_int32), ("window", C.c_int32), ("min_samples", C.c_int32), ("reserved", C.c_int32)]


class LargePlan(C.Structure):
    _fields_ = [("N", c_i64), ("n_pad", c_i64), ("world", c_i32), ("rank", c_i32), ("row_tiles", c_i64),
                ("n_blockcols", c_i64), ("n_local_blockcols", c_i64), ("local_doubles", c_i64),
                ("panel_doubles", c_i64), ("winv_doubles", c_i64), ("chunk_blocks", c_i64)]


LARGE_NB = 256
LARGE_MAX_CHUNKS = 16

# every symbol include/cngp.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "cngp_version": (C.c_int, []),
    "cngp_kernel_parse": (C.c_int, [C.c_char_p, C.POINTER(Kernel)]),
    "cngp_kernel_finalize": (C.c_int, [C.POINTER(Kernel)]),
    "cngp_default_config": (None, [C.POINTER(Config)]),
    "cngp_create": (C.c_int, [C.POINTER(Config), C.POINTER(c_vp)]),
    "cngp_destroy": (None, [c_vp]),
    "cngp_last_error": (C.c_char_p, [c_vp]),
    "cngp_sync": (C.c_int, [c_vp]),
    "cngp_set_stream": (C.c_int, [c_vp, c_vp, c_i32]),
    "cngp_set_precision": (C.c_int, [c_vp, c_i32]),
    "cngp_launch_count": (c_i64, [c_vp]),
    "cngp_set_profiling": (C.c_int, [c_vp, c_i32]),
    "cngp_profile_read": (C.c_int, [c_vp, c_i32, C.POINTER(C.c_double), C.POINTER(c_i64), c_i32]),
    "cngp_predict_batch": (C.c_int, [c_vp, C.POINTER(Kernel), c_dp, c_i64, c_dp, c_dp, c_dp, c_i64, c_i64, c_i32,
                                     c_i32, c_dp, c_dp, c_dp, c_ip, c_i32]),
    "cngp_lml_grad_batch": (C.c_int, [c_vp, C.POINTER(Kernel), c_dp, c_i64, c_dp, c_dp, c_i64, c_i32, c_dp, c_dp,
                                      c_ip, c_i32]),
    "cngp_lml_grad_windows": (C.c_int, [c_vp, C.POINTER(Kernel), c_dp, c_i64, c_ip, c_dp, c_dp, c_i64, c_i32, c_dp,
                                        c_dp, c_ip, c_i32]),
    "cngp_optimize_batch": (C.c_int, [c_vp, C.POINTER(Kernel), c_dp, c_i64, c_dp, c_dp, c_i64, c_i32, c_i32, c_dp,
                                      c_dp, c_ip]),
    "cngp_optimize_batch_mem": (C.c_int, [c_vp, C.POINTER(Kernel), c_dp, c_i64, c_dp, c_dp, c_i64, c_i32, c_i32, c_dp,
                                          c_dp, c_ip, c_i32]),
    "cngp_gp_slip_batch": (C.c_int, [c_vp, C.POINTER(Kernel), c_dp, c_i64, c_dp, c_dp, c_i64, c_i32, c_i32, c_i32,
                                     c_dp, c_dp, c_ip, c_ip]),
    "cngp_predict_ragged": (C.c_int, [c_vp, C.POINTER(Kernel), c_dp, c_i64, c_dp, c_dp, c_ip, c_i32, c_dp, c_ip, c_i32,
                                      c_i64, c_dp, c_dp, c_dp, c_ip, c_i32]),
    "cngp_lml_grad_ragged": (C.c_int, [c_vp, C.POINTER(Kernel), c_dp, c_i64, c_dp, c_dp, c_ip, c_i32, c_i64, c_dp, c_dp,
                                       c_ip, c_i32]),
    "cngp_optimize_ragged": (C.c_int, [c_vp, C.POINTER(Kernel), c_dp, c_i64, c_dp, c_dp, c_ip, c_i32, c_i64, c_i32, c_dp,
                                       c_dp, c_ip, c_i32]),
    "cngp_gp_slip_ragged": (C.c_int, [c_vp, C.POINTER(Kernel), c_dp, c_i64, c_dp, c_dp, c_ip, c_i32, c_i64, c_i32, c_i32,
                                      c_dp, c_dp, c_ip, c_ip, c_i32]),
    "cngp_zupt_lookahead_ragged": (C.c_int, [c_vp, c_dp, c_dp, c_i64, c_ip, c_i32, c_dp, c_dp, c_dp, c_dp, c_dp, c_i32,
                                             C.POINTER(StopConfig), c_ip, c_ip, c_ip, c_dp, c_dp, c_dp, c_dp, c_i32]),
    "cngp_default_stop_config": (None, [C.POINTER(StopConfig)]),
    "cngp_zupt_lookahead_batch": (C.c_int, [c_vp, c_dp, c_dp, c_i64, c_i32, c_dp, c_dp, c_dp, c_dp, c_dp, c_i32,
                                            C.POINTER(StopConfig), c_ip, c_ip, c_ip, c_dp, c_i32]),
    "cngp_zupt_lookahead_batch_ex": (C.c_int, [c_vp, c_dp, c_dp, c_i64, c_i32, c_dp, c_dp, c_dp, c_dp, c_dp, c_i32,
                                               C.POINTER(StopConfig), c_ip, c_ip, c_ip, c_dp, c_dp, c_dp, c_dp, c_i32]),
    "cngp_ekf_covariance_batch": (C.c_int, [c_vp, c_dp, c_dp, c_dp, c_dp, c_dp, c_i64, c_i32, c_i32, c_i32, c_dp, c_i32]),
    "cngp_llh_to_enu": (C.c_int, [c_vp, c_dp, c_i64, C.POINTER(StopConfig), c_dp, c_i32]),
    "cngp_ekf_context_batch": (C.c_int, [c_vp, c_dp, c_dp, c_dp, c_dp, c_i64, C.c_double, C.c_double, c_dp, c_dp, c_dp,
                                         c_i32]),
    "cngp_default_slip_config": (None, [C.POINTER(SlipConfig)]),
    "cngp_slip_record_batch": (C.c_int, [c_vp, c_dp, c_dp, c_dp, c_dp, c_dp, c_i64, c_i32, C.POINTER(SlipConfig), c_i32,
                                         c_i32, c_dp, c_dp, c_dp, c_ip, c_ip, c_ip, c_ip, c_i32]),
    "cngp_chol_large": (C.c_int, [c_vp, C.POINTER(Kernel), c_dp, c_dp, c_dp, c_i64, c_dp, c_dp, c_dp, c_dp, c_i32]),
    "cngp_large_make_plan": (C.c_int, [c_i64, c_i32, c_i32, C.POINTER(LargePlan)]),
    "cngp_large_assemble": (C.c_int, [c_vp, C.POINTER(LargePlan), C.POINTER(Kernel), c_dp, c_dp, c_dp, c_dp]),
    "cngp_large_factor_panel": (C.c_int, [c_vp, C.POINTER(LargePlan), c_dp, c_i64, c_dp, c_dp, c_dp, c_ip]),
    "cngp_large_factor_panel_ex": (C.c_int, [c_vp, C.POINTER(LargePlan), c_dp, c_i64, c_dp, c_dp, c_dp, c_ip, c_i32, c_i32]),
    "cngp_large_panel_chunks": (C.c_int, [C.POINTER(LargePlan), c_i64, C.POINTER(c_i32), C.POINTER(c_i32), C.POINTER(c_i64)]),
    "cngp_large_backsolve_finish": (C.c_int, [c_vp, C.POINTER(LargePlan), c_dp, c_i64, c_dp, c_dp, c_dp]),
    "cngp_large_backsolve_apply": (C.c_int, [c_vp, C.POINTER(LargePlan), c_dp, c_i64, c_dp, c_dp]),
    "cngp_large_copy_back": (C.c_int, [c_vp, C.POINTER(LargePlan), c_dp, c_i64, c_dp]),
    "cngp_large_update_part": (C.c_int, [c_vp, C.POINTER(LargePlan), c_dp, c_i64, c_dp, c_i64, c_i64, c_i32, c_i32]),
    "cngp_large_update": (C.c_int, [c_vp, C.POINTER(LargePlan), c_dp, c_i64, c_dp, c_i64, c_i64]),
    "cngp_large_reduce": (C.c_int, [c_vp, C.POINTER(LargePlan), c_dp, c_dp, c_ip, c_dp, c_dp]),
    "cngp_large_backsolve_step": (C.c_int, [c_vp, C.POINTER(LargePlan), c_dp, c_dp, c_i64, c_dp, c_dp]),
    "cngp_large_matvec": (C.c_int, [c_vp, C.POINTER(Kernel), c_dp, c_dp, c_dp, c_i64, c_dp]),
    "cngp_large_predict_sizes": (C.c_int, [C.POINTER(LargePlan), c_i64, c_i64, C.POINTER(c_i64), C.POINTER(c_i64),
                                           C.POINTER(c_i64)]),
    "cngp_large_predict_assemble": (C.c_int, [c_vp, C.POINTER(LargePlan), C.POINTER(Kernel), c_dp, c_dp, c_dp, c_i64, c_dp]),
    "cngp_large_predict_panel": (C.c_int, [c_vp, C.POINTER(LargePlan), c_dp, c_dp, c_dp, c_i64, c_i64, c_dp, c_dp]),
    "cngp_large_predict_update": (C.c_int, [c_vp, C.POINTER(LargePlan), c_dp, c_i64, c_i64, c_dp, c_i64, c_i64]),
    "cngp_large_predict_finish": (C.c_int, [c_vp, C.POINTER(LargePlan), C.POINTER(Kernel), c_dp, c_dp, c_dp, c_dp, c_i64,
                                            c_dp, c_dp, c_dp]),
    "cngp_chol_large_predict": (C.c_int, [c_vp, C.POINTER(Kernel), c_dp, c_dp, c_dp, c_i64, c_dp, c_i64, c_dp, c_dp, c_dp,
                                          c_dp, c_dp, c_i32]),
    "cngp_large_grad_sizes": (C.c_int, [C.POINTER(LargePlan), C.POINTER(c_i64), C.POINTER(c_i64), C.POINTER(c_i64)]),
    "cngp_large_grad_begin": (C.c_int, [c_vp, C.POINTER(LargePlan), c_dp]),
    "cngp_large_grad_panel": (C.c_int, [c_vp, C.POINTER(LargePlan), c_dp, c_dp, c_dp, c_i64, c_dp]),
    "cngp_large_grad_update": (C.c_int, [c_vp, C.POINTER(LargePlan), c_dp, c_i64, c_dp, c_i64, c_i64]),
    "cngp_large_grad_contract": (C.c_int, [c_vp, C.POINTER(LargePlan), C.POINTER(Kernel), c_dp, c_dp, c_dp, c_dp, c_dp]),
    "cngp_large_grad_finish": (C.c_int, [c_vp, C.POINTER(LargePlan), C.POINTER(Kernel), c_dp, c_dp]),
    "cngp_chol_large_grad": (C.c_int, [c_vp, C.POINTER(Kernel), c_dp, c_dp, c_dp, c_i64, c_dp, c_dp, c_dp, c_dp, c_i32]),
}

LARGE_GRAD_STRIDE = MAX_PARAMS + 1   # row length of the gradient parts (cngp_large_grad_sizes)

_lib = None


def load() -> C.CDLL:
    """Load libcngp.so, declaring every entry point.  Raises RuntimeError if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m corenav_gp_b200.build` (nvcc, sm_100a). "
            "corenav_gp_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
