"""ctypes binding of the C-ABI in include/spmm_b200.h (libspmm_b200.so, built in-tree).

The library is the product: there is no Python or CPU fallback. Importing this
module without the built library raises, and every call on a machine without a
CUDA device fails with the library's own error (SPMM_ERR_CUDA).
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SPMM_B200_LIB") or os.path.join(HERE, "libspmm_b200.so")  # override: diagnostic builds only

SPMM_OK, SPMM_ERR_INVALID, SPMM_ERR_CUDA, SPMM_ERR_NOMEM, SPMM_ERR_UNSUPPORTED = range(5)
KERNEL_AUTO, KERNEL_ROWS, KERNEL_MERGE, KERNEL_TILED, KERNEL_STREAM, KERNEL_BSR = 0, 1, 2, 6, 8, 9
KERNELS = {"auto": KERNEL_AUTO, "rows": KERNEL_ROWS, "merge": KERNEL_MERGE, "tiled": KERNEL_TILED, "stream": KERNEL_STREAM,
           "bsr": KERNEL_BSR}


class SpmmError(RuntimeError):
    """Non-zero spmm_status; mirrors the reference's only error convention (std::runtime_error)."""

    def __init__(self, status: int, message: str):
        super().__init__(f"spmm_b200 status {status}: {message}")
        self.status = status


_p = C.c_void_p
_i = C.c_int
_ll = C.c_longlong
_ull = C.c_ulonglong
_d = C.c_double
_pi = C.POINTER(C.c_int)
_pll = C.POINTER(C.c_longlong)
_pd = C.POINTER(C.c_double)

# name -> (restype, argtypes). Every symbol include/spmm_b200.h declares is listed here;
# tests/test_cabi_symbols.py checks the header, this table and the built library agree.
PROTOTYPES = {
    "spmm_last_error": (C.c_char_p, []),
    "spmm_last_kernel_name": (C.c_char_p, []),
    "spmm_version": (_i, []),
    "spmm_device_count": (_i, [_pi]),
    "spmm_device_info": (_i, [_i, _pi, _pll, _pll]),
    "spmm_csr_create_host": (_i, [_i, _i, _i, _ll, _p, _p, _p, C.POINTER(_p)]),
    "spmm_csr_create_device": (_i, [_i, _i, _i, _ll, _p, _p, _p, _i, C.POINTER(_p)]),
    "spmm_csr_create_host64": (_i, [_i, _i, _i, _ll, _p, _p, _p, C.POINTER(_p)]),
    "spmm_csr_create_device64": (_i, [_i, _i, _i, _ll, _p, _p, _p, _i, C.POINTER(_p)]),
    "spmm_csr_device_ptrs64": (_i, [_p, C.POINTER(_p), C.POINTER(_p), C.POINTER(_p)]),
    "spmm_csr_download64": (_i, [_p, _p, _p, _p]),
    "spmm_csr_from_coo_host": (_i, [_i, _i, _i, _ll, _p, _p, _p, _i, C.POINTER(_p)]),
    "spmm_csr_from_coo_device": (_i, [_i, _i, _i, _ll, _p, _p, _p, _i, C.POINTER(_p)]),
    "spmm_mm_read": (_i, [C.c_char_p, _pi, _pi, _pll, _pi, C.POINTER(_p), C.POINTER(_p), C.POINTER(_p)]),
    "spmm_mm_free": (None, [_p, _p, _p]),
    "spmm_csr_from_matrix_market": (_i, [_i, C.c_char_p, C.POINTER(_p)]),
    "spmm_csr_destroy": (_i, [_p]),
    "spmm_csr_info": (_i, [_p, _pi, _pi, _pll, _pi]),
    "spmm_csr_device_ptrs": (_i, [_p, C.POINTER(_p), C.POINTER(_p), C.POINTER(_p)]),
    "spmm_csr_update_values_device": (_i, [_p, _p, _p]),
    "spmm_csr_update_values_host": (_i, [_p, _p]),
    "spmm_csr_download": (_i, [_p, _p, _p, _p]),
    "spmm_csr_schedule": (_i, [_p, _pll, _pi, _pd, _pi]),
    "spmm_csr_column_block": (_i, [_p, _i, _i, C.POINTER(_p)]),
    "spmm_csr_build_tiles": (_i, [_p, _i, _i]),
    "spmm_csr_build_tiles_for_k": (_i, [_p, _i, _i, _i]),
    "spmm_csr_column_span": (_i, [_p, _pi, _pi]),
    "spmm_csr_build_bsr": (_i, [_p, _i, _pi]),
    "spmm_multiply_host_rows": (_i, [_p, _p, _i, _p, _i]),
    "spmm_multiply_host_sink": (_i, [_p, _p, _i, _p, _p, _i]),
    "spmm_fetch_c_sink": (_i, [_p, _p, _i, _i, _p, _p]),
    "spmm_host_threads": (_i, []),
    "spmm_host_parallel_for": (None, [_i, _p, _p]),
    "spmm_stage_b_rows": (_i, [_p, _p, _i, _i, _i, C.POINTER(_p), C.POINTER(_p)]),
    "spmm_csr_stream_sync": (_i, [_p]),
    "spmm_upload_dense": (_i, [_p, _p, _ll, _i, _p, _p]),
    "spmm_download_dense": (_i, [_p, _p, _ll, _i, _p, _p]),
    "spmm_fetch_c_rows": (_i, [_p, _p, _i, _i, _p]),
    "spmm_device_scratch": (_i, [_i, _i, _ll, C.POINTER(_p)]),
    "spmm_device_scratch_release": (_i, []),
    "spmm_peer_enable": (_i, [_i, _i]),
    "spmm_add_device": (_i, [_i, _p, _p, _ll, _p]),
    "spmm_copy_device": (_i, [_i, _p, _p, _ll, _p]),
    "spmm_device_sync": (_i, [_i]),
    "spmm_devices_init": (_i, [_i]),
    "spmm_device_init": (_i, [_i]),
    "spmm_fill_zero_device": (_i, [_i, _p, _ll, _p]),
    "spmm_csr_tile_info": (_i, [_p, _pi, _pi, _pi, _pi, _pd, _pd]),
    "spmm_multiply_device": (_i, [_p, _p, _i, _p, _i, _p]),
    "spmm_multiply_scatter_device": (_i, [_p, _p, _i, _i, C.POINTER(_p), _i, _p]),
    "spmm_multiply_window_device": (_i, [_p, _p, _i, _i, _i, _p, _i, _p]),
    "spmm_multiply_strided_device": (_i, [_p, _p, _i, _p, _i, _i, _i, _i, _p]),
    "spmm_multiply_host": (_i, [_p, _p, _i, _p, _i]),
    "spmm_multiply_rows_device": (_i, [_p, _i, _i, _p, _i, _p, _i, _p]),
    "spmm_multiply_rows_host": (_i, [_p, _i, _i, _p, _i, _p, _i]),
    "spmm_multiply_nnz_range_host": (_i, [_p, _ll, _ll, _i, _i, _p, _i, _p, _i]),
    "spmm_nnz_range_rows": (_i, [_p, _ll, _ll, _pi, _pi]),
    "spmm_multiply_nnz_range_device": (_i, [_p, _ll, _ll, _i, _i, _p, _i, _p, _i, _p]),
    "spmm_reduce_blocks_device": (_i, [_i, _i, C.POINTER(_p), _ll, _p, _p]),
    "spmm_partition_rows": (None, [_i, _i, _i, _pi, _pi]),
    "spmm_partition_cols": (None, [_i, _i, _i, _pi, _pi]),
    "spmm_partition_nnz": (None, [_ll, _i, _i, _pll, _pll]),
    "spmm_generate_fat_vector": (None, [_i, _i, _p]),
    "spmm_are_equal": (_i, [_p, _p, _ll, _d]),
    "spmm_gen_banded": (_i, [_i, _i, _i, _i, _ull, C.POINTER(_p)]),
    "spmm_gen_banded_rows": (_i, [_i, _i, _i, _i, _i, _i, _ull, C.POINTER(_p)]),
    "spmm_gen_rmat": (_i, [_i, _i, _ll, _d, _d, _d, _ull, C.POINTER(_p)]),
    "spmm_gen_fat_vector_device": (_i, [_i, _p, _ll, _ll, _ull, _p]),
    "spmm_tune_set": (_i, [C.c_char_p, _i]),
}

_lib = None


def lib() -> C.CDLL:
    """The loaded library; raises if it has not been built (python __graft_entry__.py build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `make -C {os.path.join(HERE, 'csrc')}` "
                "(or __graft_entry__.build()). There is no CPU fallback for this path.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(status: int) -> None:
    if status != SPMM_OK:
        raise SpmmError(status, (lib().spmm_last_error() or b"").decode())


def reduce_blocks(device: int, src_ptrs, n_elems: int, out_ptr: int, stream: int = 0) -> None:
    """out = sum of the source blocks in list order (peer buffers over NVLink allowed); spmm_reduce_blocks_device."""
    arr = (C.c_void_p * len(src_ptrs))(*[C.c_void_p(int(p)) for p in src_ptrs])
    check(lib().spmm_reduce_blocks_device(device, len(src_ptrs), arr, n_elems, C.c_void_p(out_ptr), C.c_void_p(stream)))


def partition_rows(n_rows: int, n_ranks: int, rank: int) -> tuple[int, int]:
    """RowWise.cpp:26-29."""
    b, e = C.c_int(), C.c_int()
    lib().spmm_partition_rows(n_rows, n_ranks, rank, C.byref(b), C.byref(e))
    return b.value, e.value


def partition_cols(k: int, n_ranks: int, rank: int) -> tuple[int, int]:
    """ColumnWise.cpp:25-28."""
    b, e = C.c_int(), C.c_int()
    lib().spmm_partition_cols(k, n_ranks, rank, C.byref(b), C.byref(e))
    return b.value, e.value


def partition_nnz(nnz: int, n_ranks: int, rank: int) -> tuple[int, int]:
    """NonZeroElement.cpp:24-39."""
    b, e = C.c_longlong(), C.c_longlong()
    lib().spmm_partition_nnz(nnz, n_ranks, rank, C.byref(b), C.byref(e))
    return b.value, e.value


def tune(key: str, value: int) -> None:
    check(lib().spmm_tune_set(key.encode(), int(value)))
