"""ctypes loader for libbmsparse_b200.so (the C ABI declared in include/bmsparse_b200.h).

There is no CPU fallback: if the shared library is missing or fails to load, importing any operator
raises.  Build it with `python -c "import __graft_entry__ as g; g.build()"` or `make -C
bmsparse_spgemm_spmv_b200/csrc`.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BMSP_LIB_PATH") or os.path.join(_HERE, "lib", "libbmsparse_b200.so")   # override: A/B runs of two builds

F16, F32 = 0, 1
HOST, DEVICE = 0, 1

STATUS = {0: "OK", 1: "INVALID", 2: "CUDA", 3: "UNSORTED", 4: "DUPLICATE", 5: "IO", 6: "TOO_LARGE",
          7: "UNSUPPORTED", 8: "RANGE"}


class BmspError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"bmsparse_b200: {STATUS.get(code, code)}: {msg}")
        self.code = code


class View(C.Structure):
    _fields_ = [("num_rows", C.c_int32), ("num_cols", C.c_int32), ("nnz", C.c_int64), ("block_num", C.c_int64),
                ("keys", C.c_void_p), ("bmps", C.c_void_p), ("offsets", C.c_void_p), ("values", C.c_void_p),
                ("offsets_len", C.c_int64), ("dtype", C.c_int32), ("transposed", C.c_int32),
                ("num_block_rows", C.c_int32), ("block_row_ptr", C.c_void_p), ("block_col", C.c_void_p),
                ("block_row_val", C.c_void_p)]


class SpgemmInfo(C.Structure):
    _fields_ = [("symbolic_ms", C.c_float), ("numeric_ms", C.c_float), ("total_ms", C.c_float),
                ("candidate_pairs", C.c_int64), ("surviving_pairs", C.c_int64), ("c_blocks", C.c_int64),
                ("c_nnz", C.c_int64), ("numeric_path", C.c_int32), ("count_ms", C.c_float), ("fill_ms", C.c_float)]


HALO_MAX = 8


class HaloDesc(C.Structure):
    _fields_ = [("n_push", C.c_int32), ("push_lo", C.c_int32 * HALO_MAX), ("push_hi", C.c_int32 * HALO_MAX),
                ("push_dst", C.c_void_p * HALO_MAX), ("n_peer", C.c_int32), ("peer_flag", C.c_void_p * HALO_MAX),
                ("my_flag", C.c_void_p * HALO_MAX), ("scratch", C.c_void_p), ("own_col_lo", C.c_int32), ("own_col_hi", C.c_int32)]


class SpgemmOpts(C.Structure):
    _fields_ = [("mode", C.c_int32), ("tc_version", C.c_int32), ("verbose", C.c_int32), ("numeric_path", C.c_int32),
                ("brow_begin", C.c_int32), ("brow_end", C.c_int32), ("brow_range_set", C.c_int32)]


# every symbol include/bmsparse_b200.h declares (tests check the library exports each one)
SYMBOLS = ["bmsp_abi_version", "bmsp_last_error", "bmsp_device_info", "bmsp_create_from_csr", "bmsp_create_from_coo",
           "bmsp_create_from_mtx", "bmsp_create_from_arrays", "bmsp_destroy", "bmsp_get", "bmsp_download",
           "bmsp_to_coo", "bmsp_compare", "bmsp_to_csr", "bmsp_compare_csr", "bmsp_create_from_coo_ex", "bmsp_create_from_mtx_ex", "bmsp_spmv", "bmsp_spmv_host", "bmsp_spmv_bytes", "bmsp_spgemm", "bmsp_block_transpose",
           "bmsp_partition_block_rows", "bmsp_slice_block_rows", "bmsp_debug_pair_bitmap", "bmsp_spmv_halo", "bmsp_halo_push",
           "bmsp_halo_status", "bmsp_peer_alloc", "bmsp_peer_open", "bmsp_peer_close", "bmsp_peer_free", "bmsp_set_values",
           "bmsp_set_values_csr", "bmsp_spgemm_plan_create", "bmsp_spgemm_numeric", "bmsp_spgemm_plan_bytes", "bmsp_spgemm_plan_destroy",
           "bmsp_matrix_transpose", "bmsp_add", "bmsp_debug_spmv_plan", "bmsp_debug_spmv_shapes"]

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} not built; there is no CPU fallback (run __graft_entry__.build())")
        _lib = C.CDLL(LIB_PATH)
        _lib.bmsp_last_error.restype = C.c_char_p
        for name in SYMBOLS:
            getattr(_lib, name)
    return _lib


def check(code: int) -> None:
    if code != 0:
        raise BmspError(code, lib().bmsp_last_error().decode(errors="replace"))
