"""New values for a resident matrix (spmm_csr_update_values_device / _host, DeviceCSR.update_values, the strategies'
update_values): the handle keeps its schedule and tile layout, and every kernel multiplies with the new values."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import sparsematrixmultiplicationmpi_b200 as spmm
from sparsematrixmultiplicationmpi_b200 import _cabi, generators as gen
from conftest import REL_TOL, assert_close_rel, random_csr

gpu = pytest.mark.gpu


# ---------------------------------------------------------------- helpers (as in test_gpu_parity.py)
def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def banded_csr(seed, n, mean_len, half_band, planes=(0,), long_row=None, empty_every=0):
    """FEM-like rows: columns cluster in windows of +-half_band around i + p for each plane offset p."""
    rng = np.random.default_rng(seed)
    lens = rng.poisson(mean_len, n)
    if empty_every:
        lens[::empty_every] = 0
    if long_row is not None:
        lens[n // 2] = long_row
    rowptr = np.concatenate(([0], np.cumsum(lens))).astype(np.int32)
    rows = np.repeat(np.arange(n), lens)
    centre = rows + rng.choice(np.asarray(planes), rows.size)
    col = np.clip(centre + rng.integers(-half_band, half_band + 1, rows.size), 0, n - 1).astype(np.int32)
    for i in range(n):
        col[rowptr[i]:rowptr[i + 1]].sort()
    return rowptr, col, 0.5 + rng.random(rows.size)


TILED_SHAPES = {
    # name: (n, mean_len, half_band, planes, long_row, empty_every); fem_hub_empty: a split 900-long row, empty rows
    "fem3": (6000, 22, 12, (-700, 0, 700), None, 0),
    "fem_hub_empty": (5003, 18, 20, (-300, 0, 300), 900, 7),
    "narrow": (3001, 5, 3, (0,), None, 3),
    "tiny": (5, 3, 2, (0,), None, 0),
}


def new_values(seed, nnz):
    """Mixed signs, so that a stale value cannot hide in a sum."""
    return np.random.default_rng(seed).standard_normal(nnz)


def multiply(A, dB, k, kernel):
    dC = torch.full((A.n_rows, k), np.nan, dtype=torch.float64, device="cuda")
    A.multiply(dB.data_ptr(), k, dC.data_ptr(), kernel, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return dC.cpu().numpy()


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def tensor_over(ptr, n):
    """A float64 CUDA tensor over memory the library owns (no copy)."""
    class View:
        __cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (int(ptr), False), "version": 3}
    return torch.as_tensor(View(), device="cuda")


def device_vals_ptr(A):
    p = C.c_void_p()
    _cabi.check(_cabi.lib().spmm_csr_device_ptrs(A.handle, None, None, C.byref(p)))
    return p.value


@pytest.fixture
def tuning_reset():
    _cabi.tune("reset", 0)
    yield
    _cabi.tune("reset", 0)


# ---------------------------------------------------------------- 1. tiled kernel, bit for bit
def _tiled_update_case(oracle, rp, ci, v0, v1, k, T, BR, tune):
    n = len(rp) - 1
    for key, val in tune.items():
        _cabi.tune(key, val)
    B = np.random.default_rng(k).integers(1, 101, (n, k)).astype(np.float64)
    dB = dev(B)
    m0, m1 = spmm.SparseMatrix(v0, ci, rp, n, n), spmm.SparseMatrix(v1, ci, rp, n, n)
    with spmm.DeviceCSR.from_host(m0, 0) as A, spmm.DeviceCSR.from_host(m1, 0) as F:
        try:
            info = A.build_tiles(T, BR, k)
        except _cabi.SpmmError as e:
            assert e.status == _cabi.SPMM_ERR_UNSUPPORTED  # this tile shape needs more shared memory than an SM has
            pytest.skip("tile shape does not fit")
        assert F.build_tiles(T, BR, k) == info
        c0 = multiply(A, dB, k, "tiled")
        A.update_values(dev(v1))  # device form
        c1 = multiply(A, dB, k, "tiled")
        assert A.tile_info() == info
        fresh = multiply(F, dB, k, "tiled")
        assert np.array_equal(bits(c1), bits(fresh))
        assert_close_rel(c1, oracle.spmm(rp, ci, v1, B, k), rp, ci, v1, B)
        A.update_values(np.ascontiguousarray(v0))  # and back through the host form
        assert np.array_equal(bits(multiply(A, dB, k, "tiled")), bits(c0))


@gpu
@pytest.mark.parametrize("shape", list(TILED_SHAPES))
@pytest.mark.parametrize("k", [2, 8, 16, 32, 48, 64])
@pytest.mark.parametrize("T,BR", [(8, 4), (64, 32), (248, 16)])
def test_tiled_update_bitwise(oracle, tuning_reset, shape, k, T, BR):
    """k-tiles of 8 (k <= 8) and 16 columns, chunks shared by 1 / 2 / 4 CTAs (k < 32, 32 and 48, 64)."""
    n, mean, hb, planes, long_row, ee = TILED_SHAPES[shape]
    rp, ci, v0 = banded_csr(31, n, mean, hb, planes, long_row, ee)
    _tiled_update_case(oracle, rp, ci, v0, new_values(1, v0.size), k, T, BR, {})


@gpu
@pytest.mark.parametrize("tune", [{"tiled.group": 1}, {"tiled.group": 3, "tiled.stride": 600}, {"tiled.thr": 1},
                                  {"tiled.thr": 100}])
@pytest.mark.parametrize("T,BR", [(8, 4), (64, 32), (248, 16)])
@pytest.mark.parametrize("k", [16, 64])
def test_tiled_update_walking_orders_and_box_thresholds(oracle, tuning_reset, tune, T, BR, k):
    """Walking orders (tiles one far band apart in turn, or as they lie) and box thresholds (all boxes / all single rows)."""
    n, mean, hb, planes, long_row, ee = TILED_SHAPES["fem_hub_empty"]
    rp, ci, v0 = banded_csr(37, n, mean, hb, planes, long_row, ee)
    _tiled_update_case(oracle, rp, ci, v0, new_values(2, v0.size), k, T, BR, tune)


# ---------------------------------------------------------------- 2. values edited in place
@gpu
def test_in_place_edit_through_device_ptrs(oracle):
    n, mean, hb, planes, long_row, ee = TILED_SHAPES["fem_hub_empty"]
    rp, ci, v0 = banded_csr(41, n, mean, hb, planes, long_row, ee)
    v1, k = new_values(3, v0.size), 32
    B = np.random.default_rng(5).integers(1, 101, (n, k)).astype(np.float64)
    dB = dev(B)
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(v0, ci, rp, n, n), 0) as A, \
            spmm.DeviceCSR.from_host(spmm.SparseMatrix(v1, ci, rp, n, n), 0) as F:
        assert A.build_tiles(64, 16, k)["rows_per_tile"] == 64 and F.build_tiles(64, 16, k)["rows_per_tile"] == 64
        multiply(A, dB, k, "tiled")
        own = tensor_over(device_vals_ptr(A), A.nnz)
        own.copy_(dev(v1))
        A.update_values(own)  # the handle's own array: only the layout is refreshed
        assert device_vals_ptr(A) == own.data_ptr()
        assert np.array_equal(bits(multiply(A, dB, k, "tiled")), bits(multiply(F, dB, k, "tiled")))
        assert A.download().values.tobytes() == v1.tobytes()


@gpu
def test_in_place_edit_of_a_borrowed_handle(oracle):
    n, mean, hb, planes, long_row, ee = TILED_SHAPES["fem3"]
    rp, ci, v0 = banded_csr(43, n, mean, hb, planes, long_row, ee)
    v1, k = new_values(4, v0.size), 16
    B = np.random.default_rng(6).integers(1, 101, (n, k)).astype(np.float64)
    dB = dev(B)
    d_rp, d_ci, d_v = dev(rp), dev(ci), dev(v0)
    h = C.c_void_p()
    _cabi.check(_cabi.lib().spmm_csr_create_device(0, n, n, v0.size, d_rp.data_ptr(), d_ci.data_ptr(), d_v.data_ptr(), 0,
                                                   C.byref(h)))
    with spmm.DeviceCSR(h.value, owner=(d_rp, d_ci, d_v)) as A, \
            spmm.DeviceCSR.from_host(spmm.SparseMatrix(v1, ci, rp, n, n), 0) as F:
        assert A.build_tiles(64, 16, k)["rows_per_tile"] == 64 and F.build_tiles(64, 16, k)["rows_per_tile"] == 64
        multiply(A, dB, k, "tiled")
        d_v.copy_(dev(v1))  # the caller rewrites its own array ...
        A.update_values(d_v)  # ... and says so
        assert np.array_equal(bits(multiply(A, dB, k, "tiled")), bits(multiply(F, dB, k, "tiled")))


# ---------------------------------------------------------------- 3. CSR kernels and the partial forms
@gpu
@pytest.mark.parametrize("layout", [False, True])
def test_csr_kernels_and_partial_forms_read_new_values(tuning_reset, layout):
    n = 4001
    rp, ci, v0 = banded_csr(47, n, 16, 14, (-400, 0, 400), long_row=300, empty_every=7)
    v1 = new_values(5, v0.size)
    m0, m1 = spmm.SparseMatrix(v0, ci, rp, n, n), spmm.SparseMatrix(v1, ci, rp, n, n)
    stream = torch.cuda.current_stream().cuda_stream
    with spmm.DeviceCSR.from_host(m0, 0) as A, spmm.DeviceCSR.from_host(m1, 0) as F:
        if layout:
            assert A.build_tiles(64, 16, 16)["rows_per_tile"] == 64
        A.update_values(v1)  # host form

        def both(fn, shape):
            out = []
            for H in (A, F):
                d = torch.full(shape, np.nan, dtype=torch.float64, device="cuda")
                fn(H, d)
                torch.cuda.synchronize()
                out.append(d.cpu().numpy())
            assert np.array_equal(bits(out[0]), bits(out[1]))

        for k in (1, 2, 4, 8, 16):
            dB = dev(np.random.default_rng(k).integers(1, 101, (n, k)).astype(np.float64))
            kernels = ("rows", "merge") + (("stream",) if k <= 8 else ())
            for kernel in kernels:
                both(lambda H, d: H.multiply(dB.data_ptr(), k, d.data_ptr(), kernel, stream), (n, k))
            both(lambda H, d: H.multiply_rows(1000, 3001, dB.data_ptr(), k, d.data_ptr(), "rows", stream), (2001, k))
            first, last = A.nnz_range_rows(12345, 40000)
            both(lambda H, d: H.multiply_nnz_range(12345, 40000, first, last, dB.data_ptr(), k, d.data_ptr(), "rows", stream),
                 (last - first + 1, k))
            lo, hi = A.column_span()
            both(lambda H, d: H.multiply_window(dB[lo:hi + 1].data_ptr(), lo, hi + 1 - lo, k, d.data_ptr(), "rows", stream),
                 (n, k))
            both(lambda H, d: H.multiply_scatter(dB.data_ptr(), k, [d.data_ptr()], "merge", stream), (n, k))
        dB = dev(np.random.default_rng(9).integers(1, 101, (n, 12)).astype(np.float64))
        both(lambda H, d: H.multiply_strided(dB.data_ptr(), 12, d.data_ptr(), 12, 4, 6, "rows", stream), (n, 12))


# ---------------------------------------------------------------- 4. AUTO keeps its state
@gpu
def test_auto_layout_survives_updates(oracle, tuning_reset):
    n, nc, r, c, v, sym = gen.cop20k_A_shaped(n=30_000, nnz=600_000, nx=20, ny=25, seed=7)
    with spmm.DeviceCSR.from_coo_host(n, nc, r, c, v, sym) as A0:
        host = A0.download()
    rp, ci = host.rowPtr, host.colIndices
    k = 64
    B = np.random.default_rng(11).integers(1, 101, (n, k)).astype(np.float64)
    dB = dev(B)
    with spmm.DeviceCSR.from_host(host, 0) as A:
        for _ in range(20):
            multiply(A, dB, k, "auto")
            if _cabi.lib().spmm_last_kernel_name() == b"spmm_tiled_kernel":
                break
        assert _cabi.lib().spmm_last_kernel_name() == b"spmm_tiled_kernel"
        info = A.tile_info()
        for step in range(3):
            v1 = np.abs(new_values(20 + step, host.nnz)) + 0.5
            A.update_values(v1 if step % 2 else dev(v1))  # host and device forms in turn
            got = multiply(A, dB, k, "auto")
            assert _cabi.lib().spmm_last_kernel_name() == b"spmm_tiled_kernel" and A.tile_info() == info
            assert_close_rel(got, oracle.spmm(rp, ci, v1, B, k), tol=REL_TOL)
        # k = 8 makes AUTO rebuild its layout (8-column k-tile) from the CSR values, which are the new ones
        v2 = np.abs(new_values(30, host.nnz)) + 0.5
        A.update_values(v2)
        B8 = np.random.default_rng(12).integers(1, 101, (n, 8)).astype(np.float64)
        got = multiply(A, dev(B8), 8, "auto")
        assert A.tile_info()["rows_per_tile"] > 0
        assert_close_rel(got, oracle.spmm(rp, ci, v2, B8, 8), tol=REL_TOL)
    # an explicit non-default layout keeps its (T, BR) across updates
    with spmm.DeviceCSR.from_host(host, 0) as A:
        info = A.build_tiles(32, 8, k)
        assert (info["rows_per_tile"], info["box_rows"]) == (32, 8)
        for step in range(2):
            v1 = np.abs(new_values(40 + step, host.nnz)) + 0.5
            A.update_values(v1)
            got = multiply(A, dB, k, "auto")
            assert A.tile_info() == info and _cabi.lib().spmm_last_kernel_name() == b"spmm_tiled_kernel"
            assert_close_rel(got, oracle.spmm(rp, ci, v1, B, k), tol=REL_TOL)


# ---------------------------------------------------------------- 5. bits
@gpu
@pytest.mark.parametrize("form", ["host", "device"])
def test_bits_survive(form):
    n, mean, hb, planes, long_row, ee = TILED_SHAPES["fem_hub_empty"]
    rp, ci, v0 = banded_csr(53, n, mean, hb, planes, long_row, ee)
    v1 = new_values(6, v0.size)
    raw = v1.view(np.uint64)
    raw[0:3] = [0x8000000000000000, 0x0000000000000001, 0x000FFFFFFFFFFFFF]  # -0.0, the smallest and largest subnormal
    raw[3:5] = [0x7FF8000000000123, 0xFFF4000000000042]  # a quiet NaN with a payload, a negative signalling one
    raw[-1] = 0x8000000000000000
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(v0, ci, rp, n, n), 0) as A:
        A.build_tiles(64, 16, 16)
        A.update_values(v1 if form == "host" else dev(v1))
        torch.cuda.synchronize()
        assert A.download().values.tobytes() == v1.tobytes()


# ---------------------------------------------------------------- 6. independence and edge cases
@gpu
def test_handles_are_independent_and_empty_update_is_a_no_op():
    n, mean, hb, planes, long_row, ee = TILED_SHAPES["fem3"]
    rp, ci, v0 = banded_csr(59, n, mean, hb, planes, long_row, ee)
    m0, k = spmm.SparseMatrix(v0, ci, rp, n, n), 16
    dB = dev(np.random.default_rng(7).integers(1, 101, (n, k)).astype(np.float64))
    with spmm.DeviceCSR.from_host(m0, 0) as A, spmm.DeviceCSR.from_host(m0, 0) as Bh:
        A.build_tiles(64, 16, k)
        Bh.build_tiles(64, 16, k)
        before = multiply(Bh, dB, k, "tiled")
        A.update_values(new_values(8, v0.size))
        A.update_values(dev(new_values(9, v0.size)))
        assert Bh.download().values.tobytes() == v0.tobytes()
        assert np.array_equal(bits(multiply(Bh, dB, k, "tiled")), bits(before))
        assert m0.values.tobytes() == v0.tobytes()
    empty = spmm.SparseMatrix(np.empty(0), np.empty(0, np.int32), np.zeros(7, np.int32), 6, 6)
    with spmm.DeviceCSR.from_host(empty, 0) as E:
        E.update_values(np.empty(0))
        E.update_values(torch.empty(0, dtype=torch.float64, device="cuda"))
        _cabi.check(_cabi.lib().spmm_csr_update_values_device(E.handle, None, None))
        _cabi.check(_cabi.lib().spmm_csr_update_values_host(E.handle, None))


@gpu
def test_host_form_after_many_host_multiplies(oracle):
    n, mean, hb, planes, long_row, ee = TILED_SHAPES["fem_hub_empty"]
    rp, ci, v0 = banded_csr(61, n, mean, hb, planes, long_row, ee)
    v1, k = new_values(10, v0.size), 24
    B = np.random.default_rng(8).integers(1, 101, (n, k)).astype(np.float64)
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(v0, ci, rp, n, n), 0) as A, \
            spmm.DeviceCSR.from_host(spmm.SparseMatrix(v1, ci, rp, n, n), 0) as F:
        A.build_tiles(64, 16, k)
        F.build_tiles(64, 16, k)
        for _ in range(12):
            A.multiply_host(B, k, "tiled")
        A.update_values(v1)
        assert np.array_equal(bits(A.multiply_host(B, k, "tiled")), bits(F.multiply_host(B, k, "tiled")))
        assert_close_rel(A.multiply_host(B, k, "auto"), oracle.spmm(rp, ci, v1, B, k), rp, ci, v1, B)


# ---------------------------------------------------------------- 7. errors
@gpu
def test_rejected_updates_leave_the_handle_working(oracle):
    n, mean, hb, planes, long_row, ee = TILED_SHAPES["fem3"]
    rp, ci, v0 = banded_csr(67, n, mean, hb, planes, long_row, ee)
    k = 16
    B = np.random.default_rng(9).integers(1, 101, (n, k)).astype(np.float64)
    dB = dev(B)
    ref = oracle.spmm(rp, ci, v0, B, k)
    lib = _cabi.lib()

    def still_works(A):
        assert_close_rel(multiply(A, dB, k, "tiled"), ref, rp, ci, v0, B)

    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(v0, ci, rp, n, n), 0) as A:
        A.build_tiles(64, 16, k)
        assert lib.spmm_csr_update_values_device(A.handle, None, None) == _cabi.SPMM_ERR_INVALID
        assert lib.spmm_csr_update_values_host(A.handle, None) == _cabi.SPMM_ERR_INVALID
        assert lib.spmm_csr_update_values_device(None, dB.data_ptr(), None) == _cabi.SPMM_ERR_INVALID
        still_works(A)
        wide = np.repeat(v0, 2)
        bad = [v0[:-1], v0.astype(np.float32), wide[::2], v0.reshape(1, -1), list(v0), torch.from_numpy(v0),
               dev(v0).float(), dev(wide)[::2], dev(v0)[:-1]]
        for values in bad:
            with pytest.raises(ValueError):
                A.update_values(values)
            still_works(A)
        if torch.cuda.device_count() > 1:
            with pytest.raises(ValueError):
                A.update_values(torch.from_numpy(v0).to("cuda:1"))
            still_works(A)
    d_rp, d_ci, d_v = dev(rp), dev(ci), dev(v0)
    h = C.c_void_p()
    _cabi.check(lib.spmm_csr_create_device(0, n, n, v0.size, d_rp.data_ptr(), d_ci.data_ptr(), d_v.data_ptr(), 0,
                                           C.byref(h)))
    with spmm.DeviceCSR(h.value, owner=(d_rp, d_ci, d_v)) as A:
        A.build_tiles(64, 16, k)
        foreign = dev(new_values(11, v0.size))
        for call in (lambda: A.update_values(foreign), lambda: A.update_values(np.ascontiguousarray(v0))):
            with pytest.raises(_cabi.SpmmError) as e:
                call()
            assert e.value.status == _cabi.SPMM_ERR_INVALID
            still_works(A)
        assert d_v.cpu().numpy().tobytes() == v0.tobytes()  # the lent array was not written


# ---------------------------------------------------------------- 8. strategies on one GPU
@gpu
def test_strategies_update_values_on_one_gpu(oracle):
    rp, ci, v0 = random_csr(19, 3000, 3000, 15, long_row=4000, empty_every=7, positive=True)
    v1 = 0.5 + np.random.default_rng(12).random(v0.size)
    m0, m1 = spmm.SparseMatrix(v0, ci, rp, 3000, 3000), spmm.SparseMatrix(v1, ci, rp, 3000, 3000)
    B = np.random.default_rng(2).integers(1, 101, (3000, 16)).astype(np.float64)
    seq = oracle.spmm(rp, ci, v1, B, 16)
    eng = spmm.CudaCompute()
    dB = dev(B)
    row = spmm.RowWise.from_host(eng, m0, 16)
    blk = spmm.ColumnBlocks.from_host(eng, m0, 16)
    slabs = spmm.ColumnSlabs.from_host(eng, m0, 16)
    nz = spmm.NonZeroRanges.from_host(eng, m0, 16)
    for plan in (row, blk, slabs, nz):
        plan.update_values(m1)
    assert_close_rel(row.run(dB).cpu().numpy(), seq, tol=REL_TOL)
    assert_close_rel(blk.run(blk.local_B(dB)).cpu().numpy(), seq, tol=REL_TOL)
    assert_close_rel(slabs.run(dB).cpu().numpy(), seq, tol=REL_TOL)
    assert_close_rel(nz.run(dB).cpu().numpy(), seq, tol=REL_TOL)
    rp2, ci2, v2 = random_csr(19, 3000, 3000, 15, long_row=4001, empty_every=7, positive=True)
    other = spmm.SparseMatrix(v2, ci2, rp2, 3000, 3000)  # one non-zero more
    for plan in (row, blk, slabs, nz):
        with pytest.raises(ValueError):
            plan.update_values(other)
        with pytest.raises(ValueError):
            plan.update_values(spmm.SparseMatrix(v1, ci, rp, 3000, 3001))


# ---------------------------------------------------------------- 9. multi-rank slicing on CPU (gloo)
class SlicingEngine:
    """Test-only engine on CPU tensors (arithmetic by the oracle): a shard is its host SparseMatrix; update_values
    replaces its values and records what each shard was handed."""

    def __init__(self):
        from test_strategies_gloo import OracleCompute
        self.inner = OracleCompute()
        self.device = self.inner.device
        self.handed = []

    def __getattr__(self, name):
        return getattr(self.inner, name)

    def update_values(self, A, values):
        values = np.asarray(values)
        assert values.dtype == np.float64 and values.ndim == 1 and values.size == A.nnz
        self.handed.append(values.copy())
        m = A.m
        A.m = spmm.SparseMatrix(values.copy(), m.colIndices, m.rowPtr, m.numRows, m.numCols)


def _slicing_worker(rank, world, port, case, results):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        seed, n, mean, k, long_row, empty_every = case
        rowptr, colidx, v0 = random_csr(seed, n, n, mean, long_row=long_row, empty_every=empty_every)
        v1 = np.random.default_rng(seed + 1).standard_normal(v0.size)
        m0, m1 = spmm.SparseMatrix(v0, colidx, rowptr, n, n), spmm.SparseMatrix(v1, colidx, rowptr, n, n)
        Bt = torch.from_numpy(np.random.default_rng(seed).integers(1, 101, (n, k)).astype(np.float64))
        eng = SlicingEngine()
        out = {}
        for name, cls in (("row", spmm.RowWise), ("colblk", spmm.ColumnBlocks), ("colslab", spmm.ColumnSlabs),
                          ("nnz", spmm.NonZeroRanges)):
            plan = cls.from_host(eng, m0, k)
            plan.update_values(m1)
            want = cls.from_host(eng, m1, k).A.m  # what the rank uploads when the plan is made from m1
            assert eng.handed[-1].tobytes() == want.values.tobytes(), name
            assert plan.A.m.values.tobytes() == want.values.tobytes(), name
            out[name] = plan.run(plan.local_B(Bt) if name == "colblk" else Bt)
        if rank == 0:
            results.update({name: t.numpy().copy() for name, t in out.items()})
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world,case", [
    (2, (71, 90, 6, 4, None, 5)),
    (2, (72, 64, 4, 3, 500, 7)),  # hub row cut by the non-zero range boundary
    (3, (73, 50, 3, 5, 400, 0)),  # hub row spanning all three ranks
])
def test_strategies_update_values_slices_world(oracle, world, case):
    mgr = mp.Manager()
    results = mgr.dict()
    mp.spawn(_slicing_worker, args=(world, _free_port(), case, results), nprocs=world, join=True)
    seed, n, mean, k, long_row, empty_every = case
    rowptr, colidx, v0 = random_csr(seed, n, n, mean, long_row=long_row, empty_every=empty_every)
    v1 = np.random.default_rng(seed + 1).standard_normal(v0.size)
    B = np.random.default_rng(seed).integers(1, 101, (n, k)).astype(np.float64)
    seq = oracle.spmm(rowptr, colidx, v1, B, k, "seq")
    assert np.array_equal(results["row"], oracle.spmm(rowptr, colidx, v1, B, k, "row", world))
    assert np.array_equal(results["colslab"], oracle.spmm(rowptr, colidx, v1, B, k, "col", world))
    assert np.array_equal(results["nnz"], oracle.spmm(rowptr, colidx, v1, B, k, "nnz", world))
    scale = np.abs(v1).max() * 100 * max(np.diff(rowptr).max(), 1)
    assert np.allclose(results["colblk"], seq, rtol=1e-12, atol=1e-12 * scale)


def test_update_values_needs_a_plan_made_from_the_host_matrix():
    rowptr, colidx, v0 = random_csr(74, 20, 20, 3)
    m = spmm.SparseMatrix(v0, colidx, rowptr, 20, 20)
    eng = SlicingEngine()
    plan = spmm.RowWise(eng, 20, 2, eng.upload(m))
    with pytest.raises(ValueError):
        plan.update_values(m)
