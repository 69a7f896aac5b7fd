"""ctypes binding of libcosmogp_b200.so (include/cosmogp_b200.h).

The library is the ONLY compute path of this package: there is no CPU fallback.
Loading fails loudly when the shared object is missing, and every compute call
fails loudly when no CUDA device is usable.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcosmogp_b200.so")

CGP_AMP_ON_AUTOCOV = 1
CGP_MEAN_TEMPLATE = 2
CGP_GRID_UNIFORM = 4
CGP_SMALL_MAX_N = 224
CGP_LOO_PLAIN = 0
CGP_LOO_RECENTER = 1

_i64 = C.c_int64
_int = C.c_int
_dbl = C.c_double
_ptr = C.c_void_p
_u32 = C.c_uint

# name -> (restype, argtypes); mirrors include/cosmogp_b200.h one to one
_BATCH = [_i64, _ptr, _int]                      # n_obj, off, dim   (host flavour)
_BATCH_DEV = [_i64, _ptr, _int, _int]            # n_obj, off, max_n, dim
_HYP = [_ptr, _dbl, _dbl, _u32]                  # hyp, nugget, floor, flags
SIGNATURES = {
    "cgp_version": (_int, []),
    "cgp_last_error": (C.c_char_p, []),
    "cgp_device_count": (_int, []),
    "cgp_fp64_peak": (_int, [_int, C.POINTER(_dbl)]),
    "cgp_launch_count": (_i64, []),
    "cgp_ll_batched_dev": (_int, _BATCH_DEV + [_ptr] * 4 + _HYP + [_ptr, _ptr, _ptr]),
    "cgp_ll_total_dev": (_int, _BATCH_DEV + [_ptr] * 4 + _HYP + [_ptr, _ptr, _ptr, _ptr, _ptr]),
    "cgp_ll_batched_host": (_int, _BATCH + [_ptr] * 4 + _HYP + [_ptr, _ptr, C.POINTER(_dbl)]),
    "cgp_ll_objhyp_dev": (_int, _BATCH_DEV + [_ptr] * 4 + [_ptr, _ptr, _dbl, _dbl, _u32, _ptr, _i64, _ptr, _ptr, _ptr]),
    "cgp_large_ll_ws_doubles": (_i64, [_i64]),
    "cgp_large_ll_objhyp_dev": (_int, [_i64, _ptr, _int] + [_ptr] * 4 + [_ptr, _ptr, _dbl, _dbl, _u32, _ptr, _i64, _ptr, _ptr,
                                                                       _ptr, _i64, _ptr]),
    "cgp_streamer_create": (_int, [_i64, _int, _i64, _int, _int, C.POINTER(_ptr)]),
    "cgp_streamer_destroy": (None, [_ptr]),
    "cgp_streamer_set_mean_spline": (_int, [_ptr, _ptr, _ptr, _int]),
    "cgp_streamer_run": (_int, [_ptr, _i64] + [_ptr] * 4 + [_ptr, _dbl, _dbl, _u32] + [_ptr, _ptr] + [_ptr] * 4
                         + [C.POINTER(_dbl), C.POINTER(_i64), C.POINTER(_i64)]),
    "cgp_spline_mean_dev": (_int, [_ptr, _ptr, _int, _ptr, _i64, _ptr, _i64, _ptr, _ptr, _ptr]),
    "cgp_grid_is_uniform": (_int, [_ptr, _i64, _ptr]),
    "cgp_streamer_schedule": (_i64, [_i64, _i64, _int, _ptr, _i64]),
    "cgp_moments_dev": (_int, [_ptr, _i64, _dbl, _ptr, _ptr]),
    "cgp_fit_objects_dev": (_int, _BATCH_DEV + [_ptr] * 4 + [_ptr, _int, _dbl, _dbl, _u32, _dbl, _dbl, _int, _int] + [_ptr] * 5),
    "cgp_predict_objhyp_dev": (_int, _BATCH_DEV + [_ptr] * 4 + [_ptr, _ptr, _dbl, _dbl, _u32] + [_ptr, _ptr, _i64, _ptr, _ptr, _ptr, _ptr, _ptr]),
    "cgp_loo_objhyp_dev": (_int, _BATCH_DEV + [_ptr] * 4 + [_ptr, _ptr, _dbl, _dbl, _u32] + [_int] + [_ptr] * 4 + [_ptr, _ptr]),
    "cgp_predict_batched_dev": (_int, _BATCH_DEV + [_ptr] * 4 + _HYP + [_ptr, _ptr, _i64, _ptr, _ptr, _ptr, _ptr, _ptr]),
    "cgp_step_batched_dev": (_int, _BATCH_DEV + [_ptr] * 4 + _HYP + [_ptr, _ptr, _i64, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr]),
    "cgp_predict_batched_host": (_int, _BATCH + [_ptr] * 4 + _HYP + [_ptr, _ptr, _i64, _ptr, _ptr, _ptr, _ptr]),
    "cgp_factor_ws_doubles": (_i64, [_int]),
    "cgp_factor_batched_dev": (_int, _BATCH_DEV + [_ptr] * 4 + _HYP + [_ptr, _ptr, _ptr, _ptr]),
    "cgp_predict_factored_dev": (_int, _BATCH_DEV + [_ptr, _ptr, _dbl, _u32, _ptr, _ptr, _ptr, _ptr, _i64, _ptr, _ptr, _ptr, _ptr]),
    "cgp_loo_batched_dev": (_int, _BATCH_DEV + [_ptr] * 4 + _HYP + [_int] + [_ptr] * 4 + [_ptr, _ptr]),
    "cgp_loo_batched_host": (_int, _BATCH + [_ptr] * 4 + _HYP + [_int] + [_ptr] * 4 + [_ptr]),
    "cgp_covariance_batched_dev": (_int, _BATCH_DEV + [_ptr] * 2 + _HYP + [_ptr, _ptr, _ptr, _i64, _ptr, _ptr, _ptr, _ptr]),
    "cgp_matrices_batched_dev": (_int, _BATCH_DEV + [_ptr] * 2 + _HYP + [_ptr, _ptr, _ptr, _ptr, _ptr]),
    "cgp_set_nccl_library": (_int, [C.c_char_p]),
    "cgp_shard_ranges": (_int, [_i64, _ptr, _int, _ptr]),
    "cgp_ctx_create": (_int, [_int, _ptr, C.POINTER(_ptr)]),
    "cgp_ctx_destroy": (None, [_ptr]),
    "cgp_ctx_info": (_int, [_ptr, C.POINTER(_int), C.POINTER(_int)]),
    "cgp_ctx_gather_f64": (_int, [_ptr, _ptr, _ptr, _ptr, _int]),
    "cgp_ctx_allreduce_sum_f64": (_int, [_ptr, _ptr, _i64]),
    "cgp_ctx_batch_create": (_int, [_ptr, _i64, _ptr, _int, _ptr, _ptr, _ptr, _ptr, C.POINTER(_ptr)]),
    "cgp_ctx_batch_destroy": (None, [_ptr]),
    "cgp_ctx_batch_ranges": (_int, [_ptr, _ptr]),
    "cgp_ctx_batch_ll": (_int, [_ptr, _ptr, _dbl, _dbl, _u32, C.POINTER(_dbl), _ptr, _ptr]),
    "cgp_ctx_batch_predict": (_int, [_ptr, _ptr, _dbl, _dbl, _u32, _ptr, _i64, _ptr, _ptr, _ptr, _ptr, _ptr, _int]),
    "cgp_ctx_batch_loo": (_int, [_ptr, _ptr, _dbl, _dbl, _u32, _int, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _int]),
    "cgp_pad128": (_i64, [_i64]),
    "cgp_cov_matrix_dev": (_int, [_int, _ptr, _i64, _ptr, _i64, _ptr] + _HYP + [_ptr, _i64, _i64, _i64, _ptr]),
    "cgp_potrf_dev": (_int, [_ptr, _i64, _i64, _ptr, _ptr, _ptr]),
    "cgp_potrs_dev": (_int, [_ptr, _i64, _i64, _ptr, _ptr, _int, _ptr]),
    "cgp_large_solve_dev": (_int, [_ptr, _i64, _i64, _i64, _ptr, _ptr, _ptr, _ptr, _ptr]),
    "cgp_large_predict_dev": (_int, [_ptr, _i64, _i64, _i64, _int, _ptr, _ptr, _ptr, _dbl, _u32,
                                     _ptr, _i64, _ptr, _ptr, _ptr, _ptr, _i64, _ptr]),
    "cgp_large_loo_dev": (_int, [_ptr, _i64, _i64, _i64, _int, _ptr, _ptr, _ptr] + _HYP + [_int, _ptr, _ptr, _i64]
                          + [_ptr] * 4 + [_ptr]),
    "cgp_trsm_rows_dev": (_int, [_ptr, _i64, _i64, _ptr, _i64, _i64, _ptr]),
    "cgp_gemm_nt_dev": (_int, [_ptr, _i64, _ptr, _i64, _ptr, _i64, _i64, _i64, _i64, _dbl, _dbl, _int, _ptr]),
}

_lib = None


class CosmogpB200Error(RuntimeError):
    pass


def lib():
    """Load (once) and return the ctypes handle.  No fallback: a missing or unloadable
    library is an error the caller sees."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CosmogpB200Error(
                "%s not found: build it with `python -m cosmogp_b200.build` (nvcc, sm_100a). "
                "cosmogp_b200 has no CPU fallback." % LIB_PATH)
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)      # AttributeError if the header and the .so disagree
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def last_error():
    return lib().cgp_last_error().decode("utf-8", "replace")


def check(rc, what):
    """rc < 0 -> raise; rc >= 0 -> number of non-positive-definite objects."""
    if rc < 0:
        raise CosmogpB200Error("%s failed (%d): %s" % (what, rc, last_error()))
    return rc


def require_device():
    n = lib().cgp_device_count()
    if n <= 0:
        raise CosmogpB200Error("no CUDA device visible (%s); cosmogp_b200 has no CPU fallback"
                               % (last_error() if n < 0 else "device count 0"))
    return n


def hptr(a):
    """Host pointer of a C-contiguous numpy array (None -> NULL)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data


def f64(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def fp64_peak(kind=1):
    out = _dbl(0.0)
    check(lib().cgp_fp64_peak(kind, C.byref(out)), "cgp_fp64_peak")
    return out.value
