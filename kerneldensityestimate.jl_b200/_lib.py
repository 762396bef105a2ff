"""ctypes binding of libkdeb200.so (include/kdeb200.h).  There is NO CPU fallback: if the CUDA
library is missing this module raises at import of the first symbol."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("KDEB200_SO") or os.path.join(_HERE, "libkdeb200.so")

f64p = C.POINTER(C.c_double)
i64p = C.POINTER(C.c_int64)
u8p = C.POINTER(C.c_uint8)
tree_t = C.c_void_p

# name -> (restype, argtypes); kept in sync with include/kdeb200.h (tests/test_abi.py checks it)
allreduce_fn = C.CFUNCTYPE(C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int), C.c_void_p)
allreduce_v_fn = C.CFUNCTYPE(C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int), C.c_int, C.c_void_p)

SIGNATURES = {
    "kdeb200_last_error": (C.c_char_p, []),
    "kdeb200_version": (C.c_int, []),
    "kdeb200_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "kdeb200_init": (C.c_int, [C.c_int]),
    "kdeb200_init_multi": (C.c_int, [C.c_int]),
    "kdeb200_init_multi_devices": (C.c_int, [C.POINTER(C.c_int), C.c_int]),
    "kdeb200_multi_count": (C.c_int, [C.POINTER(C.c_int)]),
    "kdeb200_shutdown": (C.c_int, []),
    "kdeb200_device_props": (C.c_int, [C.POINTER(C.c_int)] * 4 + [C.POINTER(C.c_size_t)]),
    "kdeb200_tree_create": (C.c_int, [C.c_int, C.c_int64, f64p, f64p, f64p, i64p, i64p, i64p, C.POINTER(tree_t)]),
    "kdeb200_tree_create_eval": (C.c_int, [C.c_int, C.c_int64, f64p, f64p, f64p, i64p, C.POINTER(tree_t)]),
    "kdeb200_tree_destroy": (C.c_int, [tree_t]),
    "kdeb200_tree_info": (C.c_int, [tree_t, C.POINTER(C.c_int), i64p, C.POINTER(C.c_int), i64p]),
    "kdeb200_tree_build_host": (C.c_int, [C.c_int, C.c_int64, f64p, f64p, f64p, f64p, f64p, f64p, f64p, f64p,
                                          i64p, i64p, i64p, i64p, i64p]),
    "kdeb200_gibbs": (C.c_int, [C.POINTER(tree_t), C.c_int, C.c_int64, C.c_int, C.c_int, u8p, f64p, C.c_int64, f64p,
                                C.c_int64, C.c_uint64, C.c_int64, C.c_int64, f64p, i64p, i64p]),
    "kdeb200_gibbs_device": (C.c_int, [C.POINTER(tree_t), C.c_int, C.c_int64, C.c_int, C.c_int, u8p, C.c_void_p,
                                       C.c_int64, C.c_void_p, C.c_int64, C.c_uint64, C.c_int64, C.c_int64,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "kdeb200_product_kde": (C.c_int, [C.POINTER(tree_t), C.c_int, C.c_int64, C.c_int, C.c_int, u8p, C.c_uint64, f64p, i64p, f64p,
                                      C.POINTER(C.c_int)]),
    "kdeb200_gibbs_sizes": (C.c_int, [C.POINTER(tree_t), C.c_int, C.c_int, C.POINTER(C.c_int), i64p, i64p, i64p]),
    "kdeb200_philox_streams": (C.c_int, [C.c_uint64, C.c_int64, C.c_int64, C.c_int64, f64p, f64p]),
    "kdeb200_eval": (C.c_int, [tree_t, f64p, C.c_int64, C.c_int, C.c_int, f64p]),
    "kdeb200_eval_device": (C.c_int, [tree_t, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "kdeb200_loo_entropy": (C.c_int, [tree_t, f64p, f64p]),
    "kdeb200_loo_partial": (C.c_int, [tree_t, f64p, C.c_int64, C.c_int64, f64p, C.POINTER(C.c_int)]),
    "kdeb200_kde_lcv": (C.c_int, [C.c_int, C.c_int64, f64p, f64p, C.POINTER(C.c_int)]),
    "kdeb200_kde_lcv_sharded": (C.c_int, [C.c_int, C.c_int64, f64p, C.c_int64, C.c_int64, allreduce_fn, C.c_void_p, f64p,
                                          C.POINTER(C.c_int)]),
    "kdeb200_kde_lcv_sharded_v": (C.c_int, [C.c_int, C.c_int64, f64p, C.c_int64, C.c_int64, allreduce_v_fn, C.c_void_p, f64p,
                                            C.POINTER(C.c_int)]),
    "kdeb200_eval_marginals": (C.c_int, [tree_t, f64p, C.c_int64, f64p]),
    "kdeb200_sample": (C.c_int, [tree_t, C.c_int64, C.c_uint64, f64p, f64p, f64p, i64p]),
    "kdeb200_set_pruning": (C.c_int, [C.c_int]),
    "kdeb200_set_gibbs_precision": (C.c_int, [C.c_int]),
    "kdeb200_gibbs_f32_slow_draws": (C.c_int, [C.POINTER(C.c_ulonglong)]),
    "kdeb200_gibbs_exact_redone": (C.c_int, [C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]),
    "kdeb200_gibbs_exact_bound_probe": (C.c_int, [C.POINTER(tree_t), C.c_int, C.c_int, C.c_int, C.c_int, f64p, f64p, C.c_int,
                                                  f64p, C.c_int64]),
    "kdeb200_pruned_stats": (C.c_int, [f64p, i64p]),
    "kdeb200_pipe_peak": (C.c_int, [C.c_int, C.c_int, f64p, f64p]),
    "kdeb200_dfma_probe": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, f64p]),
    "kdeb200_last_kernel_ms": (C.c_int, [f64p, C.POINTER(C.c_int)]),
}

_LIB = None


class KDEError(RuntimeError):
    """Mirror of the reference's ErrorException (error(...)): every nonzero C return code."""


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            raise KDEError("libkdeb200.so is not built (%s): run `python __graft_entry__.py build`; "
                           "there is no CPU fallback" % SO_PATH)
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB


def check(rc):
    if rc != 0:
        raise KDEError(lib().kdeb200_last_error().decode("utf-8", "replace") or ("kdeb200 error %d" % rc))


def fptr(a):
    return None if a is None else a.ctypes.data_as(f64p)


def iptr(a):
    return None if a is None else a.ctypes.data_as(i64p)


def as_f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)
