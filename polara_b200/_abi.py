"""ctypes binding of ``libpolara_b200.so`` (the C-ABI declared in include/polara_b200.h).

There is no CPU fallback: if the library is missing or no sm_100 device is
present, every product entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_LIB = None
_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libpolara_b200.so")

OK, EINVAL, ENOMEM, ECUDA, ENOTIMPL = 0, 1, 2, 3, 4

i64, i32, f64 = C.c_int64, C.c_int, C.c_double
ptr = C.c_void_p



class CsrView(C.Structure):
    """``pb200_csr_view`` of include/polara_b200.h."""
    _fields_ = [("n_rows", i64), ("n_cols", i64), ("nnz", i64), ("indptr", ptr), ("indices", ptr), ("values", ptr),
                ("n_panels", C.c_int32), ("panel_cols", i64), ("panel_ptr_host", ptr)]


# name -> argtypes (after the leading ctx pointer unless noted)
_SIGNATURES = {
    "pb200_version": ([], C.c_int),
    "pb200_ctx_create": ([C.c_int, ptr, C.POINTER(ptr)], C.c_int),
    "pb200_ctx_destroy": ([ptr], C.c_int),
    "pb200_ctx_set_stream": ([ptr, ptr], C.c_int),
    "pb200_last_error": ([ptr], C.c_char_p),
    "pb200_ctx_sync": ([ptr], C.c_int),
    "pb200_debug_dump": ([ptr], C.c_int),
    "pb200_set_score_kernel": ([ptr, C.c_int], C.c_int),
    "pb200_get_stats": ([ptr, C.POINTER(C.c_uint64)], C.c_int),
    "pb200_set_reduce_hook": ([ptr, ptr, ptr], C.c_int),
    "pb200_set_bound_hook": ([ptr, ptr, ptr], C.c_int),
    "pb200_set_spmm_kernel": ([ptr, C.c_int], C.c_int),
    "pb200_set_prune": ([ptr, C.c_int], C.c_int),
    "pb200_spmm_csr": ([ptr, C.POINTER(CsrView), ptr, i64, ptr, i64, C.c_int], C.c_int),
    "pb200_coo_to_csr": ([ptr, i64, i64, i64, ptr, i64, ptr, i64, ptr, C.c_int, C.c_int, C.c_int, ptr, ptr, ptr, C.POINTER(i64)],
                         C.c_int),
    "pb200_topk_dense": ([ptr, ptr, C.c_int, i64, i64, i64, ptr, ptr, C.c_int, ptr, ptr], C.c_int),
    "pb200_downvote_dense": ([ptr, ptr, C.c_int, i64, i64, i64, ptr, ptr, i64], C.c_int),
    "pb200_shift_i64": ([ptr, ptr, i64, i64], C.c_int),
    "pb200_csr_block_columns": ([ptr, i64, i64, i64, ptr, ptr, ptr, i64, C.c_int, ptr, ptr, ptr, ptr], C.c_int),
    "pb200_rsvd_csr": ([ptr, C.POINTER(CsrView), C.POINTER(CsrView), C.c_int, C.c_int, C.c_int, f64, f64, C.c_uint64,
                        ptr, i64, ptr, ptr, i64, C.POINTER(f64)], C.c_int),
    "pb200_spmm": ([ptr, i64, i64, i64, ptr, ptr, ptr, ptr, i64, ptr, i64, C.c_int], C.c_int),
    "pb200_csr_transpose": ([ptr, i64, i64, i64, ptr, ptr, ptr, ptr, ptr, ptr], C.c_int),
    "pb200_rescale": ([ptr, i64, i64, i64, ptr, ptr, ptr, f64, f64], C.c_int),
    "pb200_rsvd": ([ptr, i64, i64, i64, ptr, ptr, ptr, ptr, ptr, ptr, C.c_int, C.c_int, C.c_int, f64,
                    C.c_uint64, ptr, i64, ptr, ptr, i64, C.POINTER(C.c_int)], C.c_int),
    "pb200_tall_svd": ([ptr, ptr, i64, C.c_int, i64, C.c_int, ptr, ptr, i64, ptr], C.c_int),
    "pb200_score_topk": ([ptr, ptr, i64, ptr, i64, i64, i64, C.c_int, ptr, ptr, C.c_int, i64, ptr, ptr], C.c_int),
    "pb200_score_topk_cands": ([ptr, ptr, i64, ptr, i64, i64, i64, C.c_int, ptr, ptr, C.c_int, i64, ptr], C.c_int),
    "pb200_merge_cands_fill": ([ptr, ptr, C.c_int, i64, i64, C.c_int, ptr, i64, ptr, i64, C.c_int, i64, ptr, ptr, ptr, ptr],
                               C.c_int),
    "pb200_fill_empty_cands": ([ptr, ptr, i64], C.c_int),
    "pb200_merge_cands": ([ptr, ptr, C.c_int, i64, C.c_int, ptr, ptr], C.c_int),
    "pb200_gather_dot": ([ptr, ptr, i64, i64, ptr, i64, i64, C.c_int, ptr, ptr, i64, ptr], C.c_int),
    "pb200_score_dense": ([ptr, ptr, i64, ptr, i64, i64, i64, C.c_int, ptr, i64], C.c_int),
    "pb200_ttm": ([ptr, i64, i64, ptr, ptr, ptr, ptr, ptr, C.c_int, i64, ptr, C.c_int, i64, ptr, i64], C.c_int),
    "pb200_ttm_reduce": ([ptr, C.c_int, i64, ptr, ptr, ptr, ptr, ptr, C.c_int, i64, ptr, C.c_int, i64, ptr, i64],
                         C.c_int),
    "pb200_coo_group": ([ptr, i64, i64, ptr, ptr, ptr, ptr, ptr, ptr, ptr, ptr], C.c_int),
    "pb200_sgd_plan": ([ptr, i64, i64, i64, ptr, ptr, ptr, ptr, C.c_int, ptr, ptr, ptr, ptr, ptr, ptr, ptr, ptr], C.c_int),
    "pb200_sgd_epoch": ([ptr, C.c_int, ptr, ptr, ptr, ptr, ptr, ptr, ptr, i64, ptr, i64, C.c_int, f64, f64,
                         C.POINTER(f64)], C.c_int),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

# int (*pb200_reduce_fn)(void* user, void* dev_ptr, int64_t count, int dtype)
REDUCE_FN = C.CFUNCTYPE(C.c_int, ptr, ptr, i64, C.c_int)


class LibraryMissing(RuntimeError):
    pass


def lib_path():
    return _LIB_PATH


def load():
    """Load the shared library (once) and attach the prototypes."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(_LIB_PATH):
        raise LibraryMissing(
            "%s not found -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(polara_b200 has no CPU fallback)" % _LIB_PATH)
    lib = C.CDLL(_LIB_PATH)
    for name, (argtypes, restype) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = ABI drift, fail loudly
        fn.argtypes = argtypes
        fn.restype = restype
    _LIB = lib
    return lib


_EXC = {EINVAL: ValueError, ENOMEM: MemoryError, ECUDA: RuntimeError, ENOTIMPL: NotImplementedError}


def check(ctx_handle, status, where=""):
    if status == OK:
        return
    msg = ""
    if ctx_handle:
        raw = load().pb200_last_error(ctx_handle)
        msg = raw.decode("utf-8", "replace") if raw else ""
    raise _EXC.get(status, RuntimeError)("polara_b200 %s failed (status %d): %s" % (where, status, msg))
