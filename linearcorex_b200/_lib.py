"""ctypes binding of liblcx_b200.so (the C ABI declared in include/lcx_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, this module raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblcx_b200.so")

OK, QUICK_FAIL = 0, 1
ERR_SINGULAR, ERR_NOT_PD, ERR_MISSING = -4, -5, -6
PRECISION_FP64, PRECISION_FAST, PRECISION_FP64_SPLIT, PRECISION_FP64_SPLIT5, PRECISION_FP64_SPLIT7 = 0, 1, 2, 3, 4
PRECISIONS = {"fp64": PRECISION_FP64, "fast": PRECISION_FAST, "fp64_split": PRECISION_FP64_SPLIT,
              "fp64_split5": PRECISION_FP64_SPLIT5, "fp64_split7": PRECISION_FP64_SPLIT7}
SPLIT_DIGITS = {"fast": 3, "fp64_split": 6, "fp64_split5": 5, "fp64_split7": 7}
F32, F64 = 0, 1
GAUSS = {"standard": 0, "outliers": 1, "none": 2}

# enum lcx_array (include/lcx_b200.h)
(A_W, A_RHO, A_INVRHO, A_RHOINVRHO, A_QIJ, A_SI, A_QISI2, A_RY, A_UJ, A_GRAD, A_UPDATE, A_RDIR, A_D, A_MI, A_XZ,
 A_XY, A_X2Y, A_IXY, A_YJ2, A_IYX, A_TCS, A_TCDIRECT, A_CY, A_Y, A_SCALARS, A_COUNT) = range(26)

ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_longlong, C.c_longlong)

_p, _i, _ll, _d, _ull = C.c_void_p, C.c_int, C.c_longlong, C.c_double, C.c_ulonglong
_pd = C.POINTER(C.c_double)
_pll = C.POINTER(C.c_longlong)

# name -> (restype, argtypes): every symbol include/lcx_b200.h declares
SIGNATURES = {
    "lcx_version": (_i, []),
    "lcx_last_error": (C.c_char_p, []),
    "lcx_session_create": (_i, [C.POINTER(_p), _i, _i]),
    "lcx_session_destroy": (_i, [_p]),
    "lcx_set_stream": (_i, [_p, _p]),
    "lcx_set_allreduce": (_i, [_p, ALLREDUCE_FN, _p]),
    "lcx_peer_buffer_doubles": (_ll, [_i, _i]),
    "lcx_set_peer_allreduce": (_i, [_p, _i, _i, C.POINTER(C.c_void_p), _ll]),
    "lcx_launch_count": (_i, [_p, _pll]),
    "lcx_profile_enable": (_i, [_p, _i]),
    "lcx_profile_read": (_i, [_p, _pd, _pd, _pll, _i]),
    "lcx_profile_read_phases": (_i, [_p, _pd, _pd, _pd, _pll, _i]),
    "lcx_ld": (_ll, [_i]),
    "lcx_ldy": (_ll, [_i]),
    "lcx_workspace_doubles": (_ll, [_ll, _i, _i, _i]),
    "lcx_bind": (_i, [_p, _p, _ll, _ll, _i, _ll, _i, _p, _ll]),
    "lcx_gram_scratch_doubles": (_ll, [_p, _i]),
    "lcx_gram_build": (_i, [_p, _p, _ll, _i, _p, _ll]),
    "lcx_gram_workspace_doubles": (_ll, [_i, _i, _i]),
    "lcx_bind_gram": (_i, [_p, _p, _ll, _i, _i, _p, _ll]),
    "lcx_array_info": (_i, [_p, _i, _i, _pll, _pll, _pll, _pll]),
    "lcx_digit_planes_info": (_i, [_p, _i, _pll, C.POINTER(C.c_int), _pll, _pll, _pll, _pll, C.POINTER(C.c_int)]),
    "lcx_colstats_sum": (_i, [_p, _p, _i, _ll, _i, _ll, _i, _d, _p, _p, _p, _ll]),
    "lcx_colstats_mean": (_i, [_p, _p, _p, _p, _i]),
    "lcx_colstats_sqdev": (_i, [_p, _p, _i, _ll, _i, _ll, _i, _d, _p, _p, _p, _p, _ll]),
    "lcx_set_x_scale": (_i, [_p, _d]),
    "lcx_slice_block": (_i, [_p, _p, _ll, _ll, _ll]),
    "lcx_standardize_slice": (_i, [_p, _p, _i, _ll, _ll, _ll, _i, _d, _i, _p, _p, _p]),
    "lcx_colstats_std": (_i, [_p, _p, _p, _d, _i, _p, _i]),
    "lcx_standardize": (_i, [_p, _p, _i, _ll, _i, _ll, _i, _d, _i, _p, _p, _p, _p, _ll]),
    "lcx_colstats_scratch_doubles": (_ll, [_ll, _i]),
    "lcx_row_scale": (_i, [_p, _p, _ll, _d, _d, _p]),
    "lcx_colstats_sum_w": (_i, [_p, _p, _i, _ll, _i, _ll, _i, _d, _p, _p, _p, _ll, _p]),
    "lcx_colstats_sqdev_w": (_i, [_p, _p, _i, _ll, _i, _ll, _i, _d, _p, _p, _p, _p, _ll, _p, _p]),
    "lcx_standardize_w": (_i, [_p, _p, _i, _ll, _i, _ll, _i, _d, _i, _p, _p, _p, _p, _ll, _p]),
    "lcx_standardize_slice_w": (_i, [_p, _p, _i, _ll, _ll, _ll, _i, _d, _i, _p, _p, _p, _p]),
    "lcx_project": (_i, [_p, _p, _ll, _i, _ll, _p, _ll, _i, _p, _ll, _p, _p, _ll]),
    "lcx_project_scratch_doubles": (_ll, [_ll, _i]),
    "lcx_sig": (_i, [_p, _p, _d, _p]),
    "lcx_set_w": (_i, [_p, _p, _ll]),
    "lcx_get_w": (_i, [_p, _p, _ll]),
    "lcx_init_scale": (_i, [_p, _d]),
    "lcx_stage_rescale": (_i, [_p, _d, _d]),
    "lcx_permute_rows": (_i, [_p, C.POINTER(C.c_int)]),
    "lcx_moments_ns": (_i, [_p, _d, _i, _pd, _pd]),
    "lcx_details_ns": (_i, [_p, _pd, _pd]),
    "lcx_direction_ns": (_i, [_p, _d, _pd]),
    "lcx_trial_ns": (_i, [_p, _d, _d, _i, _pd, _pd]),
    "lcx_direction_trial_ns": (_i, [_p, _d, _d, _pd, _pd, _pd]),
    "lcx_run_stage_ns": (_i, [_p, _d, _d, _i, _i, _d, C.POINTER(C.c_int), C.POINTER(C.c_int), _pd, _pd, _pd,
                                C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "lcx_accept_trial": (_i, [_p]),
    "lcx_moments_syn": (_i, [_p, _pd, _pd]),
    "lcx_update_syn": (_i, [_p, _d, _pd, _pd]),
    "lcx_get_covariance": (_i, [_p, _i, _d, _p, _i, _i, _p, _ll]),
    "lcx_covariance_rows": (_i, [_p, _p, _p, _ll, _i, _i, _d, _p, _i, _i, _p, _ll]),
    "lcx_lowrank_scratch_doubles": (_ll, [_i, _i]),
    "lcx_lowrank_factor": (_i, [_p, _p, _p, _ll, _i, _i, _d, _p, _p, _ll, _p, _p, _p, _ll]),
    "lcx_score_scratch_doubles": (_ll, [_ll, _i, _i]),
    "lcx_score_rows": (_i, [_p, _p, _i, _ll, _i, _ll, _i, _d, _p, _p, _p, _p, _ll, _i, _p, _p, _p, _p, _p, _ll]),
    "lcx_precision_rows": (_i, [_p, _p, _ll, _i, _i, _p, _p, _i, _i, _p, _ll]),
    "lcx_lowrank_h_scratch_doubles": (_ll, [_i, _i]),
    "lcx_lowrank_factor_h": (_i, [_p, _p, _p, _ll, _i, _i, _d, _p, _p, _ll, _p, _p, _p, _ll, _p, _ll]),
    "lcx_condition_scratch_doubles": (_ll, [_ll, _i, _i]),
    "lcx_condition_rows": (_i, [_p, _p, _i, _ll, _i, _ll, _i, _d, _p, _p, _p, _ll, _i, _p, _ll, _p, _p, _p, _ll, _p, _p, _pll,
                                _p, _ll]),
    "lcx_condition_sample_scratch_doubles": (_ll, [_ll, _i, _i]),
    "lcx_condition_sample_rows": (_i, [_p, _p, _i, _ll, _i, _ll, _i, _d, _p, _p, _p, _ll, _i, _p, _ll, _p, _p, _ll, _p, _p, _ll,
                                       _ll, _ull, _ll, _i, _pll, _p, _ll]),
    "lcx_normal_fill": (_i, [_p, _ull, _i, _ll, _ll, _ll, _i, _p, _ll, _p, _ll]),
    "lcx_sample_scratch_doubles": (_ll, [_ll, _i, _i]),
    "lcx_sample_rows": (_i, [_p, _p, _p, _ll, _i, _i, _d, _p, _p, _ull, _ll, _ll, _p, _ll, _p, _ll]),
    "lcx_conditional_factor_scratch_doubles": (_ll, [_i, _i, _i]),
    "lcx_conditional_factor": (_i, [_p, _p, _p, _ll, _i, _i, _d, _p, _p, _p, _i, _p, _i, _p, _ll, _p, _ll, _p, _p, _p, _p, _ll]),
    "lcx_conditional_scratch_doubles": (_ll, [_ll, _i, _i]),
    "lcx_conditional_rows": (_i, [_p, _p, _i, _ll, _i, _ll, _i, _d, _p, _ll, _p, _p, _ll, _i, _p, _i, _p, _p, _ll, _p, _p, _p,
                                  _ll]),
    "lcx_conditional_sample_rows": (_i, [_p, _p, _i, _ll, _i, _ll, _i, _d, _p, _ll, _p, _p, _ll, _i, _p, _i, _p, _ll, _ll, _ull,
                                         _ll, _i, _p, _ll]),
    "lcx_conditional_covariance_rows": (_i, [_p, _p, _ll, _i, _i, _p, _i, _i, _p, _ll]),
    "lcx_gemm_f64": (_i, [_p, _i, _i, _i, _i, _p, _ll, _p, _ll, _p, _ll, _i, _p, _i, _p, _ll]),
    "lcx_solve_scratch_doubles": (_ll, [_i]),
    "lcx_solve": (_i, [_p, _p, _ll, _i, _p, _ll, _p, _ll, _i, _p, _ll]),
}

_lib = None


class LcxError(RuntimeError):
    pass


def load():
    """Load liblcx_b200.so and declare every prototype.  Raises if the library is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LcxError("%s is missing: run `python -m linearcorex_b200.build` (or __graft_entry__.build()); "
                       "there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    """Raise on a negative status; pass non-negative codes (OK / QUICK_FAIL) through."""
    if rc == ERR_SINGULAR:  # np.linalg.solve raises this at linearcorex.py:280 / :366
        import numpy as np
        raise np.linalg.LinAlgError("Singular matrix")
    if rc == ERR_NOT_PD:  # what np.linalg.cholesky raises on the dense covariance
        import numpy as np
        raise np.linalg.LinAlgError("Matrix is not positive definite")
    if rc < 0:
        msg = load().lcx_last_error()
        raise LcxError("%s failed (%d): %s" % (what or "lcx call", rc, msg.decode() if msg else "?"))
    return rc
