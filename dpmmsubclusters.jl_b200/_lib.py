"""ctypes binding of libdpmm_b200.so (include/dpmm_b200.h).

The shared library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a).  There is no CPU
fallback anywhere in this package: if the library is missing, or the machine has no CUDA device,
the calls fail loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DPMM_LIB_PATH") or os.path.join(_HERE, "libdpmm_b200.so")   # (override: development builds)

OK, EINVAL, ECUDA, ESTATE, ELIMIT, ENCCL = 0, -1, -2, -3, -4, -5
PRIOR_NIW, PRIOR_MULTINOMIAL = 0, 1
SAMPLER_INVERSE_CDF, SAMPLER_GUMBEL = 0, 1

_p = C.c_void_p
_i32, _i64, _u64 = C.c_int32, C.c_int64, C.c_uint64
_f32p, _f64p, _i64p, _u8p = (C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_int64),
                             C.POINTER(C.c_uint8))

# name -> (restype, argtypes); exactly the symbols include/dpmm_b200.h declares
SIGNATURES = {
    "dpmm_create": (C.c_int, [C.POINTER(_p), _f32p, _i64, _i32, _i32, _i32, _u64, _i64]),
    "dpmm_destroy": (C.c_int, [_p]),
    "dpmm_last_error": (C.c_char_p, [_p]),
    "dpmm_set_stream": (C.c_int, [_p, _p]),
    "dpmm_sync": (C.c_int, [_p]),
    "dpmm_limits": (C.c_int, [C.POINTER(_i32)]),
    "dpmm_init_labels": (C.c_int, [_p, _i32, _i32]),
    "dpmm_randomize_sublabels": (C.c_int, [_p, _i64p, _i32]),
    "dpmm_get_labels": (C.c_int, [_p, _i64p]),
    "dpmm_get_sublabels": (C.c_int, [_p, _i64p]),
    "dpmm_set_labels": (C.c_int, [_p, _i64p]),
    "dpmm_set_sublabels": (C.c_int, [_p, _i64p]),
    "dpmm_set_params_niw": (C.c_int, [_p, _i32, _f32p, _f32p, _f32p, _f32p, _f32p]),
    "dpmm_set_params_multinomial": (C.c_int, [_p, _i32, _f32p, _f32p, _f32p]),
    "dpmm_set_sampler": (C.c_int, [_p, _i32]),
    "dpmm_sample_labels": (C.c_int, [_p, _i32]),
    "dpmm_sample_sublabels": (C.c_int, [_p]),
    "dpmm_suff_stats": (C.c_int, [_p, _i64p, _i32, _i64p, _f64p, _f64p]),
    "dpmm_num_clusters": (C.c_int, [_p]),
    "dpmm_set_hyper_niw": (C.c_int, [_p, C.c_double, _f64p, C.c_double, _f64p, C.c_double]),
    "dpmm_set_hyper_multinomial": (C.c_int, [_p, _f32p, C.c_double]),
    "dpmm_posterior_step": (C.c_int, [_p, _i64p, _i32, _i32, _u8p, _i32, _i64p, _f64p, _f64p]),
    "dpmm_sample_params": (C.c_int, [_p, _i32, _i32, _i32]),
    "dpmm_params_merge": (C.c_int, [_p, _i64, _i64]),
    "dpmm_get_params_niw": (C.c_int, [_p, _i32, _f32p, _f64p, _f32p, _f32p, _f32p]),
    "dpmm_get_params_multinomial": (C.c_int, [_p, _i32, _f32p, _f32p, _f32p]),
    "dpmm_predict_niw": (C.c_int, [_p, _i32, _f32p, _f32p, _f32p, _f32p, _i64p, _f32p]),
    "dpmm_predict_multinomial": (C.c_int, [_p, _i32, _f64p, _f32p, _i64p, _f32p]),
    "dpmm_apply_split": (C.c_int, [_p, _i64p, _i64p, _i32]),
    "dpmm_apply_merge": (C.c_int, [_p, _i64p, _i64p, _i32]),
    "dpmm_remove_empty": (C.c_int, [_p, _i64p, _i32]),
    "dpmm_smart_project": (C.c_int, [_p, _i64, _f64p, _f64p, _f64p, _i64p]),
    "dpmm_smart_kmeans_iter": (C.c_int, [_p, C.c_double, C.c_double, _f64p]),
    "dpmm_smart_set_sublabels": (C.c_int, [_p, _i64]),
    "dpmm_nccl_unique_id": (C.c_int, [_p]),
    "dpmm_comm_init": (C.c_int, [_p, _p, _i32, _i32]),
    "dpmm_set_uniforms": (C.c_int, [_p, _f64p, _f64p, _u8p]),
    "dpmm_debug_loglik": (C.c_int, [_p, _i32, _f32p]),
    "dpmm_debug_tc_stats": (C.c_int, [_p, _i64p]),
    "dpmm_debug_sort": (C.c_int, [_p, C.POINTER(C.c_int32), _i64p]),
    "dpmm_debug_fused_stats": (C.c_int, [_p, _i64p]),
    "dpmm_timing_enable": (C.c_int, [_p, _i32]),
    "dpmm_timing_kinds": (C.c_int, []),
    "dpmm_timing_name": (C.c_char_p, [_i32]),
    "dpmm_timing_read": (C.c_int, [_p, _f64p, _i64p, _i32]),
    "dpmm_launch_count": (_i64, [_p]),
}

_lib = None


class DpmmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libdpmm_b200 error {code}: {msg}")
        self.code = code


def load():
    """dlopen the in-tree library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). This package has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, ctx=None):
    if rc != 0:
        msg = load().dpmm_last_error(ctx)
        raise DpmmError(rc, msg.decode() if msg else "?")
