"""ctypes binding of libcybayes_b200.so (C ABI in include/cybayes_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C cybayes_b200/csrc``.
There is deliberately no fallback: if the shared library is missing or no CUDA device is
visible, loading / context creation raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libcybayes_b200.so")

c_i32p = C.POINTER(C.c_int32)
c_f64p = C.POINTER(C.c_double)
c_i64p = C.POINTER(C.c_int64)

c_u32p = C.POINTER(C.c_uint32)
c_i8p = C.POINTER(C.c_int8)

# cb_chain_backend (native generation loop): callback table
CHAIN_BUILD_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, c_f64p, C.c_double, c_f64p, C.c_int, c_i32p, c_f64p, c_f64p)
CHAIN_EVAL_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_int, c_i32p, c_i32p, c_i32p, c_f64p, C.c_int,
                            C.POINTER(C.c_int), c_f64p)
CHAIN_RELEASE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int)
CHAIN_RATES_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_double, c_f64p)
CHAIN_BETA_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, c_f64p, C.c_int, c_f64p)
CHAIN_EIG_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, c_f64p, c_f64p, c_f64p)
CHAIN_EVAL_SITES_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_int, c_i32p, c_i32p, c_i32p, c_f64p, C.c_int,
                                  C.POINTER(C.c_int), c_f64p, c_f64p, c_f64p)


class ChainBackend(C.Structure):
    _fields_ = [("user", C.c_void_p), ("pmat_build", CHAIN_BUILD_FN), ("eval", CHAIN_EVAL_FN),
                ("snapshot_release", CHAIN_RELEASE_FN), ("site_rates", CHAIN_RATES_FN), ("f81_beta", CHAIN_BETA_FN),
                ("gtr_eig", CHAIN_EIG_FN), ("eval_sites", CHAIN_EVAL_SITES_FN)]


# name -> (restype, argtypes); mirrors include/cybayes_b200.h one to one
SIGNATURES = {
    "cb_chain_create": (C.c_int, [C.c_void_p, C.POINTER(ChainBackend)] + [C.c_int] * 10 +
                        [c_i32p, c_f64p, c_f64p, c_f64p, C.POINTER(C.c_void_p)]),
    "cb_chain_set_state": (C.c_int, [C.c_void_p, C.c_int, c_i32p, c_i32p, c_f64p, c_f64p, C.c_int, c_f64p, C.c_double,
                                     c_f64p, C.c_double, c_f64p, c_f64p]),
    "cb_chain_set_rng": (C.c_int, [C.c_void_p, c_u32p, C.c_int, c_u32p, C.c_int]),
    "cb_chain_get_rng": (C.c_int, [C.c_void_p, c_u32p, C.POINTER(C.c_int), c_u32p, C.POINTER(C.c_int)]),
    "cb_chain_run": (C.c_int, [C.c_void_p, C.c_int64, c_i8p, c_i8p, c_f64p, c_f64p, c_f64p, c_f64p]),
    "cb_chain_get_state": (C.c_int, [C.c_void_p, c_i32p, c_i32p, c_f64p, c_f64p, c_f64p, c_f64p, c_f64p, c_f64p]),
    "cb_chain_counters": (C.c_int, [C.c_void_p, c_i64p, c_i64p]),
    "cb_chain_site_lnl": (C.c_int, [C.c_void_p, c_f64p, c_f64p]),
    "cb_chain_destroy": (C.c_int, [C.c_void_p]),
    "cb_last_error": (C.c_char_p, []),
    "cb_version": (C.c_int, []),
    "cb_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "cb_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "cb_destroy": (C.c_int, [C.c_void_p]),
    "cb_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "cb_comm_init": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "cb_set_tips": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int,
                              c_f64p, C.c_int, c_f64p]),
    "cb_compress_patterns": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int64, C.c_int, c_i64p, c_i64p, c_f64p, c_i64p]),
    "cb_pmat_reserve": (C.c_int, [C.c_void_p, C.c_int]),
    "cb_pmat_upload": (C.c_int, [C.c_void_p, C.c_int, c_i32p, c_f64p]),
    "cb_pmat_download": (C.c_int, [C.c_void_p, C.c_int, c_i32p, c_f64p]),
    "cb_pmat_build": (C.c_int, [C.c_void_p, C.c_int, c_f64p, C.c_double, c_f64p, C.c_int, c_i32p, c_f64p, c_f64p]),
    "cb_eval": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_i32p, c_i32p, c_i32p, c_f64p, C.c_int,
                          C.POINTER(C.c_int), c_f64p]),
    "cb_eval_sites": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_i32p, c_i32p, c_i32p, c_f64p, C.c_int,
                                C.POINTER(C.c_int), c_f64p, c_f64p, c_f64p]),
    "cb_eval_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_i32p, c_i32p, c_i32p, c_i32p, c_f64p, c_f64p]),
    "cb_simulate": (C.c_int, [C.c_void_p, C.c_int, c_i32p, c_i32p, c_i32p, c_f64p, C.c_int, C.c_uint64, C.c_uint32,
                              C.c_int64, C.c_void_p]),
    "cb_result_wait": (C.c_int, [C.c_void_p, c_f64p]),
    "cb_snapshot_retain": (C.c_int, [C.c_void_p, C.c_int]),
    "cb_snapshot_release": (C.c_int, [C.c_void_p, C.c_int]),
    "cb_snapshot_read": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_f64p, c_i32p]),
    "cb_stats": (C.c_int, [C.c_void_p, c_i64p, c_i64p, c_i64p, c_i64p]),
    "cb_mem_info": (C.c_int, [C.c_void_p, c_i64p, c_i64p, c_i64p, c_i64p]),
    "cb_last_eval_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "cb_last_eval_main_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "cb_last_eval_info": (C.c_int, [C.c_void_p, c_i64p, c_i64p, c_i32p]),
    "cb_host_profile": (C.c_int, [C.c_void_p, c_f64p, C.c_int]),
    "cb_mark": (C.c_int, [C.c_void_p, C.c_int]),
    "cb_mark_elapsed_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "cb_sync": (C.c_int, [C.c_void_p]),
    "cb_fp64_peak": (C.c_int, [C.c_void_p, c_f64p]),
    "cb_flush_l2": (C.c_int, [C.c_void_p]),
}

CB_MODEL_JC, CB_MODEL_F81, CB_MODEL_F81_BINARY, CB_MODEL_GTR_EIG = 0, 1, 2, 3
CB_EVAL_WANT_SNAPSHOT, CB_EVAL_STORE_ROOT, CB_EVAL_NO_SYNC, CB_EVAL_FORCE_LEVELS, CB_EVAL_FORCE_WALK = 1, 2, 4, 8, 16
CB_EVAL_NO_FOLD = 32

_lib = None


class CyBayesB200Error(RuntimeError):
    pass


def load():
    """dlopen the in-tree library and declare every signature.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CyBayesB200Error(
            f"{LIB_PATH} is not built (run `python -c 'import __graft_entry__ as g; g.build()'` or "
            "`make -C cybayes_b200/csrc`); cybayes_b200 has no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise CyBayesB200Error(load().cb_last_error().decode("utf-8", "replace"))
