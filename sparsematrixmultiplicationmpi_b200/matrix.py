"""Host data model of the drop-in boundary and its device-resident counterpart.

`SparseMatrix` mirrors the reference struct (/root/reference "Source Code/MatrixDefinitions.h":14-19
plus the numRows/numCols its .cpp files rely on, utils.cpp:180-181): same field names, FP64
values, int32 indices. A `FatVector` is a C-contiguous float64 array of shape (N, k): the flat
row-major image the reference's serialize() produces (utils.cpp:216-228).

`DeviceCSR` owns the HBM copy of a SparseMatrix (an spmm_csr_t of include/spmm_b200.h) together
with its row-length schedule and, optionally, the row-block layout for large k.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _cabi


@dataclass
class SparseMatrix:
    values: np.ndarray      # float64[nnz]
    colIndices: np.ndarray  # int32[nnz]
    rowPtr: np.ndarray      # int32[numRows+1]
    numRows: int = 0
    numCols: int = 0

    def __post_init__(self):
        self.values = np.ascontiguousarray(self.values, dtype=np.float64)
        self.colIndices = np.ascontiguousarray(self.colIndices, dtype=np.int32)
        self.rowPtr = np.ascontiguousarray(self.rowPtr, dtype=np.int32)
        if self.numRows == 0 and self.rowPtr.size:
            self.numRows = int(self.rowPtr.size - 1)

    @property
    def nnz(self) -> int:
        return int(self.values.size)

    def row_block(self, begin: int, end: int) -> "SparseMatrix":
        """Rows [begin,end) with the row pointer rebased to 0 (what one rank of the row-wise strategy holds)."""
        lo, hi = int(self.rowPtr[begin]), int(self.rowPtr[end])
        return SparseMatrix(self.values[lo:hi], self.colIndices[lo:hi], self.rowPtr[begin:end + 1] - lo,
                            end - begin, self.numCols)


def as_fat_vector(v, n_rows: int | None = None, k: int | None = None) -> np.ndarray:
    """Accepts an (N,k) array or the reference's vector<vector<double>> shape (list of rows)."""
    a = np.ascontiguousarray(v, dtype=np.float64)
    if a.ndim == 1 and n_rows is not None and k is not None:
        a = a.reshape(n_rows, k)
    if a.ndim != 2:
        raise ValueError("FatVector must be 2-D (N rows of k doubles)")
    return a


class DeviceCSR:
    """An spmm_csr_t: CSR arrays resident in HBM + row-length schedule (+ optional row blocks)."""

    def __init__(self, handle: int, owner=None):
        self._h = C.c_void_p(handle)
        self._owner = owner  # keeps borrowed torch tensors alive
        nr, nc, dev, nnz = C.c_int(), C.c_int(), C.c_int(), C.c_longlong()
        _cabi.check(_cabi.lib().spmm_csr_info(self._h, C.byref(nr), C.byref(nc), C.byref(nnz), C.byref(dev)))
        self.n_rows, self.n_cols, self.nnz, self.device = nr.value, nc.value, nnz.value, dev.value

    # -- construction --
    @classmethod
    def from_host(cls, m: SparseMatrix, device: int = 0) -> "DeviceCSR":
        if m.rowPtr.size != m.numRows + 1:
            raise ValueError("rowPtr must hold numRows+1 offsets")
        h = C.c_void_p()
        _cabi.check(_cabi.lib().spmm_csr_create_host(device, m.numRows, m.numCols, m.nnz, m.rowPtr.ctypes.data,
                                                     m.colIndices.ctypes.data, m.values.ctypes.data, C.byref(h)))
        return cls(h.value)

    @classmethod
    def from_csr64(cls, rowptr, colidx, vals, n_rows: int, n_cols: int, device: int = 0, copy: bool = True) -> "DeviceCSR":
        """A CSR with 64-bit row offsets, for more than 2^31 - 1 stored entries (spmm_csr_create_host64 / _device64):
        rowptr int64[n_rows+1], colidx int32[nnz], vals float64[nnz]. C-contiguous numpy arrays are uploaded (copy is
        ignored); contiguous CUDA tensors on cuda:`device` are copied, or borrowed with copy=False (the DeviceCSR then
        keeps them alive; changing the pattern needs a new handle). The handle runs the int32 kernels on segments of rows
        (include/spmm_b200.h lists what it supports); every method works on it or raises SpmmError."""
        arrays = (rowptr, colidx, vals)
        if all(isinstance(a, np.ndarray) for a in arrays):
            ok_dtypes = [a.dtype for a in arrays] == [np.int64, np.int32, np.float64]
            ok_layout = all(a.ndim == 1 and a.flags.c_contiguous for a in arrays)
            sizes = [a.size for a in arrays]
            host = True
        else:
            import torch
            if not all(isinstance(a, torch.Tensor) and a.is_cuda and a.device.index == device for a in arrays):
                raise ValueError(f"rowptr/colidx/vals must be three numpy arrays or three CUDA tensors on cuda:{device}")
            ok_dtypes = [a.dtype for a in arrays] == [torch.int64, torch.int32, torch.float64]
            ok_layout = all(a.dim() == 1 and a.is_contiguous() for a in arrays)
            sizes = [a.numel() for a in arrays]
            host = False
        if not (ok_dtypes and ok_layout):
            raise ValueError("rowptr, colidx, vals must be contiguous 1-D int64, int32 and float64 arrays")
        if sizes[0] != n_rows + 1 or sizes[1] != sizes[2]:
            raise ValueError(f"rowptr must hold n_rows+1 = {n_rows + 1} offsets and colidx / vals the same count")
        nnz = sizes[1]
        h = C.c_void_p()
        if host:
            _cabi.check(_cabi.lib().spmm_csr_create_host64(device, n_rows, n_cols, nnz, rowptr.ctypes.data,
                                                           colidx.ctypes.data, vals.ctypes.data, C.byref(h)))
            return cls(h.value)
        _cabi.check(_cabi.lib().spmm_csr_create_device64(device, n_rows, n_cols, nnz, C.c_void_p(rowptr.data_ptr()),
                                                         C.c_void_p(colidx.data_ptr()), C.c_void_p(vals.data_ptr()),
                                                         int(bool(copy)), C.byref(h)))
        return cls(h.value, owner=None if copy else arrays)

    @classmethod
    def from_coo_host(cls, n_rows, n_cols, rows, cols, vals, symmetric=False, device: int = 0) -> "DeviceCSR":
        """The CSR assembly of readMatrixMarketFile (utils.cpp:124-181) done on the device."""
        rows = np.ascontiguousarray(rows, dtype=np.int32)
        cols = np.ascontiguousarray(cols, dtype=np.int32)
        vals = np.ascontiguousarray(vals, dtype=np.float64)
        if not (rows.size == cols.size == vals.size):
            raise ValueError("rows/cols/vals must have the same length")
        h = C.c_void_p()
        _cabi.check(_cabi.lib().spmm_csr_from_coo_host(device, n_rows, n_cols, rows.size, rows.ctypes.data,
                                                       cols.ctypes.data, vals.ctypes.data, int(bool(symmetric)),
                                                       C.byref(h)))
        return cls(h.value)

    @classmethod
    def banded(cls, n, nnz_per_row, half_bandwidth, seed=1, device=0, row_begin=0, row_end=None) -> "DeviceCSR":
        h = C.c_void_p()
        row_end = n if row_end is None else row_end
        _cabi.check(_cabi.lib().spmm_gen_banded_rows(device, n, row_begin, row_end, nnz_per_row, half_bandwidth,
                                                     seed, C.byref(h)))
        return cls(h.value)

    @classmethod
    def rmat(cls, scale, n_edges, a=0.57, b=0.19, c=0.19, seed=1, device=0) -> "DeviceCSR":
        h = C.c_void_p()
        _cabi.check(_cabi.lib().spmm_gen_rmat(device, scale, n_edges, a, b, c, seed, C.byref(h)))
        return cls(h.value)

    def column_block(self, col_begin: int, col_end: int) -> "DeviceCSR":
        h = C.c_void_p()
        _cabi.check(_cabi.lib().spmm_csr_column_block(self._h, col_begin, col_end, C.byref(h)))
        return DeviceCSR(h.value)

    # -- queries --
    @property
    def handle(self) -> C.c_void_p:
        if self._h is None:
            raise RuntimeError("DeviceCSR used after close()")
        return self._h

    def download(self) -> SparseMatrix:
        rowptr = np.empty(self.n_rows + 1, dtype=np.int32)
        colidx = np.empty(self.nnz, dtype=np.int32)
        vals = np.empty(self.nnz, dtype=np.float64)
        _cabi.check(_cabi.lib().spmm_csr_download(self.handle, rowptr.ctypes.data, colidx.ctypes.data,
                                                  vals.ctypes.data))
        return SparseMatrix(vals, colidx, rowptr, self.n_rows, self.n_cols)

    def download64(self) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """(rowptr int64, colidx int32, vals float64) of a handle with 64-bit row offsets (spmm_csr_download64)."""
        rowptr = np.empty(self.n_rows + 1, dtype=np.int64)
        colidx = np.empty(self.nnz, dtype=np.int32)
        vals = np.empty(self.nnz, dtype=np.float64)
        _cabi.check(_cabi.lib().spmm_csr_download64(self.handle, rowptr.ctypes.data, colidx.ctypes.data,
                                                    vals.ctypes.data))
        return rowptr, colidx, vals

    def schedule(self) -> dict:
        bins = (C.c_longlong * 8)()
        mx, mean, ak = C.c_int(), C.c_double(), C.c_int()
        _cabi.check(_cabi.lib().spmm_csr_schedule(self.handle, bins, C.byref(mx), C.byref(mean), C.byref(ak)))
        names = ["0", "1-2", "3-4", "5-8", "9-16", "17-32", "33-256", ">256"]
        return {"bins": dict(zip(names, list(bins))), "max_row_len": mx.value, "mean_row_len": mean.value,
                "auto_kernel": {1: "rows", 2: "merge"}.get(ak.value, str(ak.value))}

    def multiply_scatter(self, d_B: int, k: int, d_C_list, kernel: str = "auto", stream: int = 0) -> None:
        """C = A*B stored to every pointer of d_C_list (local and NVLink-mapped peer buffers): the row-wise
        strategy's gather fused into the multiply (spmm_multiply_scatter_device)."""
        arr = (C.c_void_p * len(d_C_list))(*[C.c_void_p(int(p)) for p in d_C_list])
        _cabi.check(_cabi.lib().spmm_multiply_scatter_device(self.handle, C.c_void_p(d_B), k, len(d_C_list), arr,
                                                             _cabi.KERNELS[kernel], C.c_void_p(stream)))

    def build_tiles(self, rows_per_tile: int = -1, box_rows: int = 0, k: int = 0) -> dict:
        """Row tiles with TMA-staged B rows (spmm_tiled.cu); -1 = tallest tile that fits shared memory.
        k (optional): the number of B columns the layout will mostly be used with — from 32 columns up the chunks are
        made longer and shared by 2 or 4 CTAs, each taking a group of k-tiles (what AUTO does on its own)."""
        _cabi.check(_cabi.lib().spmm_csr_build_tiles_for_k(self.handle, rows_per_tile, box_rows, k))
        return self.tile_info()

    def build_bsr(self, block_dim: int = -1) -> int:
        """View the CSR as b x b dense blocks (spmm_csr_build_bsr, spmm_bsr.cu): no copy, the values stay the handle's.
        block_dim: 2..6 checks that the pattern is exactly b-blocked (SpmmError with SPMM_ERR_UNSUPPORTED naming the first
        block row that breaks it), -1 takes the largest b that fits, 0 drops the view. Returns the block size in force
        (0: none). With a view, multiply(kernel="bsr") runs the BSR kernel and AUTO takes it where it measured faster."""
        b = C.c_int()
        _cabi.check(_cabi.lib().spmm_csr_build_bsr(self.handle, block_dim, C.byref(b)))
        return b.value

    def tile_info(self) -> dict:
        t, b, ns, mr, r, sf = C.c_int(), C.c_int(), C.c_int(), C.c_int(), C.c_double(), C.c_double()
        _cabi.check(_cabi.lib().spmm_csr_tile_info(self.handle, C.byref(t), C.byref(b), C.byref(ns), C.byref(mr),
                                                   C.byref(r), C.byref(sf)))
        return {"rows_per_tile": t.value, "box_rows": b.value, "window_slots": ns.value, "max_records": mr.value,
                "reuse": r.value, "single_fraction": sf.value}

    def nnz_range_rows(self, nnz_begin: int, nnz_end: int) -> tuple[int, int]:
        a, b = C.c_int(), C.c_int()
        _cabi.check(_cabi.lib().spmm_nnz_range_rows(self.handle, nnz_begin, nnz_end, C.byref(a), C.byref(b)))
        return a.value, b.value

    def update_values(self, values, stream: int | None = None) -> None:
        """New values for the same pattern (nnz float64 in CSR order); the schedule and the tile layout are kept, the
        values inside the layout are refreshed. Whether the pattern is the same is not checked.

        A C-contiguous numpy array goes up through the handle's pinned staging (spmm_csr_update_values_host) and the
        call returns when it is done. A contiguous CUDA tensor on the handle's device is enqueued on `stream` (default:
        the current torch stream) and not waited for (spmm_csr_update_values_device); it may be the handle's own value
        array edited in place. No reference to `values` is kept."""
        if isinstance(values, np.ndarray):
            if values.dtype != np.float64 or values.ndim != 1 or values.size != self.nnz or not values.flags.c_contiguous:
                raise ValueError(f"values must be a C-contiguous float64 array of {self.nnz} elements")
            _cabi.check(_cabi.lib().spmm_csr_update_values_host(self.handle, C.c_void_p(values.ctypes.data)))
            return
        import torch
        if not isinstance(values, torch.Tensor):
            raise ValueError("values must be a numpy array or a CUDA tensor")
        if (not values.is_cuda or values.device.index != self.device or values.dtype != torch.float64 or values.dim() != 1
                or values.numel() != self.nnz or not values.is_contiguous()):
            raise ValueError(f"values must be a contiguous float64 tensor of {self.nnz} elements on cuda:{self.device}")
        if stream is None:
            stream = torch.cuda.current_stream(values.device).cuda_stream
        _cabi.check(_cabi.lib().spmm_csr_update_values_device(self.handle, C.c_void_p(values.data_ptr()),
                                                              C.c_void_p(stream)))

    # -- multiply: device pointers (ints), everything on self.device --
    def multiply(self, d_B: int, k: int, d_C: int, kernel: str = "auto", stream: int = 0) -> None:
        _cabi.check(_cabi.lib().spmm_multiply_device(self.handle, d_B, k, d_C, _cabi.KERNELS[kernel], stream))

    def multiply_strided(self, d_B, ldb, d_C, ldc, k_begin, k_count, kernel="auto", stream=0) -> None:
        _cabi.check(_cabi.lib().spmm_multiply_strided_device(self.handle, d_B, ldb, d_C, ldc, k_begin, k_count,
                                                             _cabi.KERNELS[kernel], stream))

    def multiply_rows(self, row_begin, row_end, d_B, k, d_C_local, kernel="auto", stream=0) -> None:
        _cabi.check(_cabi.lib().spmm_multiply_rows_device(self.handle, row_begin, row_end, d_B, k, d_C_local,
                                                          _cabi.KERNELS[kernel], stream))

    def multiply_nnz_range(self, nnz_begin, nnz_end, first_row, last_row, d_B, k, d_C_local, kernel="auto",
                           stream=0) -> None:
        _cabi.check(_cabi.lib().spmm_multiply_nnz_range_device(self.handle, nnz_begin, nnz_end, first_row, last_row,
                                                               d_B, k, d_C_local, _cabi.KERNELS[kernel], stream))

    def multiply_host(self, B: np.ndarray, k: int, kernel: str = "auto", out: np.ndarray | None = None) -> np.ndarray:
        """Host buffers in, host buffer out (the call the reference-shaped entry points make).
        `out` lets a caller reuse a (pinned) result buffer instead of a fresh allocation."""
        B = as_fat_vector(B)
        if B.shape[0] < self.n_cols or B.shape[1] != k:
            raise ValueError(f"fat vector must be at least {self.n_cols} x {k}")
        if out is not None:
            if out.shape != (self.n_rows, k) or out.dtype != np.float64 or not out.flags.c_contiguous:
                raise ValueError("out must be a C-contiguous float64 array of shape (n_rows, k)")
            Cm = out
        else:
            Cm = np.empty((self.n_rows, k), dtype=np.float64)
        _cabi.check(_cabi.lib().spmm_multiply_host(self.handle, B.ctypes.data, k, Cm.ctypes.data,
                                                   _cabi.KERNELS[kernel]))
        return Cm

    def column_span(self) -> tuple[int, int]:
        """(min, max) column id stored: the rows of B this shard reads (spmm_csr_column_span); (0, -1) when empty."""
        lo, hi = C.c_int(), C.c_int()
        _cabi.check(_cabi.lib().spmm_csr_column_span(self.handle, C.byref(lo), C.byref(hi)))
        return lo.value, hi.value

    def multiply_window(self, d_B_window: int, first_row: int, n_rows: int, k: int, d_C: int, kernel: str = "auto",
                        stream: int = 0) -> None:
        """C = A*B with only the rows [first_row, first_row+n_rows) of B resident (spmm_multiply_window_device)."""
        _cabi.check(_cabi.lib().spmm_multiply_window_device(self.handle, C.c_void_p(d_B_window), first_row, n_rows, k,
                                                            C.c_void_p(d_C), _cabi.KERNELS[kernel], C.c_void_p(stream)))

    def upload_dense(self, src: np.ndarray, d_dst: int, stream: int = 0) -> None:
        """(n, k) float64 host block -> device buffer d_dst through the handle's pinned staging and the library's host
        threads (spmm_upload_dense); returns when the copy is done."""
        src = as_fat_vector(src)
        _cabi.check(_cabi.lib().spmm_upload_dense(self.handle, src.ctypes.data, src.shape[0], src.shape[1],
                                                  C.c_void_p(d_dst), C.c_void_p(stream)))

    def download_dense(self, d_src: int, n_rows: int, k: int, stream: int = 0, out: np.ndarray | None = None) -> np.ndarray:
        """Device buffer -> (n_rows, k) float64 host block (spmm_download_dense)."""
        dst = out if out is not None else np.empty((n_rows, k), dtype=np.float64)
        _cabi.check(_cabi.lib().spmm_download_dense(self.handle, C.c_void_p(d_src), n_rows, k, dst.ctypes.data,
                                                    C.c_void_p(stream)))
        return dst

    # -- lifetime --
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            _cabi.lib().spmm_csr_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
