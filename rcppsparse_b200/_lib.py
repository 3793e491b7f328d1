"""ctypes binding of libsparse_b200.so — the same C ABI (include/sparse_b200.h) that the drop-in
C++ header include/RcppSparse.h calls.  No torch types cross this boundary: plain pointers
and sizes.  Fails loudly when the library is missing; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libsparse_b200.so")

OK = 0
E_INVALID, E_CUDA, E_NOMEM, E_STRUCTURE, E_NODEVICE, E_UNSUPPORTED = -1, -2, -3, -4, -5, -6
PIN_HOST, NO_VALIDATE, NO_ROW_PLAN, LAZY_ROWS = 1, 2, 4, 8

# every symbol include/sparse_b200.h declares (tests/test_boundary.py checks header == this list == .so)
SYMBOLS = [
    "sb200_abi_version", "sb200_last_error", "sb200_device_count", "sb200_matrix_create",
    "sb200_matrix_adopt_device", "sb200_matrix_destroy", "sb200_matrix_dims", "sb200_matrix_refresh_values",
    "sb200_matrix_set_stream", "sb200_matrix_sync", "sb200_matrix_device_arrays", "sb200_col_sums",
    "sb200_row_sums", "sb200_col_means", "sb200_row_means", "sb200_spmv", "sb200_spmv_t", "sb200_transpose",
    "sb200_col_sums_dev", "sb200_row_sums_dev", "sb200_spmv_dev", "sb200_spmv_t_dev", "sb200_transpose_dev", "sb200_transpose_into",
    "sb200_vec_div_dev", "sb200_launch_count", "sb200_algorithmic_bytes", "sb200_synth_create",
    "sb200_synth_vector_dev", "sb200_matrix_download_columns", "sb200_matrix_row_path", "sb200_matrix_row_companion",
    "sb200_crossprod", "sb200_crossprod_dev", "sb200_matrix_band_companion", "sb200_matrix_layouts", "sb200_matrix_layout_bytes", "sb200_trim",
    "sb200_col_sums_in_rows", "sb200_gather_block", "sb200_spmm", "sb200_spmm_t", "sb200_spmm_dev", "sb200_spmm_t_dev",
    "sb200_col_vars", "sb200_row_vars", "sb200_col_vars_dev", "sb200_row_vars_dev",
    "sb200_sharded_create", "sb200_sharded_destroy", "sb200_sharded_info", "sb200_sharded_block", "sb200_sharded_col_sums",
    "sb200_sharded_row_sums", "sb200_sharded_col_means", "sb200_sharded_row_means", "sb200_sharded_spmv", "sb200_sharded_spmv_t", "sb200_sharded_transpose",
    "sb200_sharded_spmm", "sb200_sharded_spmm_t", "sb200_sharded_crossprod", "sb200_sharded_col_vars", "sb200_sharded_row_vars",
    "sb200_exchange_create", "sb200_exchange_connect", "sb200_exchange_destroy", "sb200_exchange_window",
    "sb200_exchange_gather", "sb200_exchange_reduce", "sb200_exchange_push_rows", "sb200_exchange_barrier", "sb200_exchange_status",
]


class SparseB200Error(RuntimeError):
    """A non-zero status from libsparse_b200 (what the C++ header rethrows as std::runtime_error)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"libsparse_b200 status {code}: {message}")
        self.code = code
        self.message = message


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m rcppsparse_b200.build` "
            "(__graft_entry__.build()).  There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u32, u64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_uint, C.c_uint64, C.c_double
    pp = C.POINTER(C.c_void_p)
    sig = {
        "sb200_abi_version": ([], C.c_int),
        "sb200_last_error": ([], C.c_char_p),
        "sb200_device_count": ([C.POINTER(C.c_int)], C.c_int),
        "sb200_matrix_create": ([vp, vp, vp, i32, i32, i64, C.c_int, u32, pp], C.c_int),
        "sb200_matrix_adopt_device": ([vp, vp, vp, i32, i32, i64, C.c_int, u32, pp], C.c_int),
        "sb200_matrix_destroy": ([vp], C.c_int),
        "sb200_matrix_dims": ([vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i64)], C.c_int),
        "sb200_matrix_refresh_values": ([vp, vp], C.c_int),
        "sb200_matrix_set_stream": ([vp, vp], C.c_int),
        "sb200_matrix_sync": ([vp], C.c_int),
        "sb200_matrix_device_arrays": ([vp, pp, pp, pp], C.c_int),
        "sb200_col_sums": ([vp, vp], C.c_int),
        "sb200_row_sums": ([vp, vp], C.c_int),
        "sb200_col_means": ([vp, vp], C.c_int),
        "sb200_row_means": ([vp, vp], C.c_int),
        "sb200_spmv": ([vp, vp, vp], C.c_int),
        "sb200_spmv_t": ([vp, vp, vp], C.c_int),
        "sb200_transpose": ([vp, vp, vp, vp], C.c_int),
        "sb200_col_sums_dev": ([vp, dbl, vp], C.c_int),
        "sb200_row_sums_dev": ([vp, dbl, vp], C.c_int),
        "sb200_spmv_dev": ([vp, vp, vp], C.c_int),
        "sb200_spmv_t_dev": ([vp, vp, vp], C.c_int),
        "sb200_transpose_dev": ([vp, pp], C.c_int),
        "sb200_transpose_into": ([vp, vp], C.c_int),
        "sb200_vec_div_dev": ([vp, vp, i64, dbl], C.c_int),
        "sb200_launch_count": ([], i64),
        "sb200_algorithmic_bytes": ([vp, C.c_char_p, C.POINTER(i64)], C.c_int),
        "sb200_synth_create": ([i32, i64, i64, u64, vp, i32, i32, vp, vp, vp, C.c_int, pp], C.c_int),
        "sb200_synth_vector_dev": ([vp, u64, i64, i64, vp], C.c_int),
        "sb200_matrix_download_columns": ([vp, i64, i64, vp, vp, vp, C.POINTER(i64)], C.c_int),
        "sb200_matrix_row_path": ([vp, C.POINTER(C.c_int)], C.c_int),
        "sb200_matrix_row_companion": ([vp, C.c_int], C.c_int),
        "sb200_matrix_band_companion": ([vp, C.c_int, C.c_int], C.c_int),
        "sb200_matrix_layouts": ([vp, C.POINTER(C.c_int)], C.c_int),
        "sb200_matrix_layout_bytes": ([vp, C.POINTER(i64)], C.c_int),
        "sb200_trim": ([C.c_int], C.c_int),
        "sb200_col_sums_in_rows": ([vp, vp, i64, C.c_int, vp], C.c_int),
        "sb200_gather_block": ([vp, vp, i64, vp, i64, vp], C.c_int),
        "sb200_spmm": ([vp, vp, i64, vp], C.c_int),
        "sb200_spmm_t": ([vp, vp, i64, vp], C.c_int),
        "sb200_spmm_dev": ([vp, vp, i64, vp], C.c_int),
        "sb200_spmm_t_dev": ([vp, vp, i64, vp], C.c_int),
        "sb200_col_vars": ([vp, vp], C.c_int),
        "sb200_row_vars": ([vp, vp], C.c_int),
        "sb200_col_vars_dev": ([vp, vp], C.c_int),
        "sb200_row_vars_dev": ([vp, vp], C.c_int),
        "sb200_sharded_create": ([vp, vp, vp, i32, i32, i64, C.c_int, vp, u32, pp], C.c_int),
        "sb200_sharded_destroy": ([vp], C.c_int),
        "sb200_sharded_info": ([vp, C.POINTER(C.c_int), vp], C.c_int),
        "sb200_sharded_block": ([vp, C.c_int, pp], C.c_int),
        "sb200_sharded_col_sums": ([vp, vp], C.c_int),
        "sb200_sharded_row_sums": ([vp, vp], C.c_int),
        "sb200_sharded_col_means": ([vp, vp], C.c_int),
        "sb200_sharded_row_means": ([vp, vp], C.c_int),
        "sb200_sharded_spmv": ([vp, vp, vp], C.c_int),
        "sb200_sharded_spmv_t": ([vp, vp, vp], C.c_int),
        "sb200_sharded_transpose": ([vp, vp, vp, vp], C.c_int),
        "sb200_sharded_spmm": ([vp, vp, i64, vp], C.c_int),
        "sb200_sharded_spmm_t": ([vp, vp, i64, vp], C.c_int),
        "sb200_sharded_crossprod": ([vp, vp], C.c_int),
        "sb200_sharded_col_vars": ([vp, vp], C.c_int),
        "sb200_sharded_row_vars": ([vp, vp], C.c_int),
        "sb200_crossprod": ([vp, vp], C.c_int),
        "sb200_crossprod_dev": ([vp, vp], C.c_int),
        "sb200_exchange_create": ([C.c_int, i64, pp, vp], C.c_int),
        "sb200_exchange_connect": ([vp, C.c_int, C.c_int, vp], C.c_int),
        "sb200_exchange_destroy": ([vp], C.c_int),
        "sb200_exchange_window": ([vp, pp, C.POINTER(i64), C.POINTER(i64)], C.c_int),
        "sb200_exchange_gather": ([vp, vp, i64, i64, i64], C.c_int),
        "sb200_exchange_reduce": ([vp, vp, i64, i64, i64, dbl], C.c_int),
        "sb200_exchange_push_rows": ([vp, vp, vp, vp, vp, vp, i32, i32, vp, vp, vp], C.c_int),
        "sb200_exchange_barrier": ([vp, vp], C.c_int),
        "sb200_exchange_status": ([vp], C.c_int),
    }
    for name in SYMBOLS:
        fn = getattr(L, name)  # AttributeError here = the .so does not export what the header declares
        fn.argtypes, fn.restype = sig[name]
    if L.sb200_abi_version() != 1:
        raise ImportError("libsparse_b200 ABI version mismatch")
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != OK:
        raise SparseB200Error(rc, lib().sb200_last_error().decode(errors="replace"))


def device_count() -> int:
    n = C.c_int(0)
    rc = lib().sb200_device_count(C.byref(n))
    return n.value if rc == OK else 0
