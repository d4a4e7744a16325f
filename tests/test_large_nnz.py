"""Handles with 64-bit row offsets (spmm_csr_create_host64 / _device64, DeviceCSR.from_csr64): the rows are cut into
segments that the int32 kernels run one after another. Small matrices are cut into many segments through the
seg.max_nnz tuning key, so that cuts fall inside every shape; one case goes past 2^31 stored entries on the device."""
import ctypes as C
import functools

import numpy as np
import pytest

import sparsematrixmultiplicationmpi_b200 as spmm
from sparsematrixmultiplicationmpi_b200 import _cabi, generators as gen
from conftest import REL_TOL, assert_close_rel, random_csr

gpu = pytest.mark.gpu

SEG = 300  # non-zeros per segment of the small handles (seg.max_nnz)

SHAPES = {
    # conftest.random_csr shapes: (seed, n_rows, n_cols, mean_len, long_row, empty_every); cop20k_small: see csr_of
    "fem_like": (2, 2500, 2500, 22, None, 0),
    "hub": (3, 1200, 1200, 6, 40000, 5),
    "empty_rows": (1, 3000, 3000, 4, None, 9),
    "single_row": (6, 1, 64, 900, None, 0),
    "rect_wide": (4, 700, 5000, 12, None, 0),
    "rect_tall": (5, 5000, 300, 3, None, 4),
    "cop20k_small": None,
}
KS = [1, 2, 3, 8, 16, 33, 64]


@functools.lru_cache(maxsize=None)
def csr_of(shape):
    """(rowptr int64, colidx int32, vals float64, n_cols) with positive values."""
    if SHAPES[shape] is None:
        import pyoracle
        n, nc, r, c, v, sym = gen.cop20k_A_shaped(n=6000, nnz=126_001, nx=20, ny=20, seed=5)
        rp, ci, va = pyoracle.Oracle().csr_from_coo(n, r, c, v, sym)
        va = np.abs(va) + 0.5
    else:
        seed, n, nc, mean, long_row, ee = SHAPES[shape]
        rp, ci, va = random_csr(seed, n, nc, mean, long_row=long_row, empty_every=ee, positive=True)
    return rp.astype(np.int64), np.ascontiguousarray(ci, dtype=np.int32), np.ascontiguousarray(va, dtype=np.float64), nc


def new_handle(rp, ci, va, nc, seg=SEG):
    _cabi.tune("seg.max_nnz", seg)
    try:
        return spmm.DeviceCSR.from_csr64(rp, ci, va, len(rp) - 1, nc)
    finally:
        _cabi.tune("reset", 0)


@pytest.fixture(scope="module")
def handle():
    """handle(shape): one segmented handle per shape for the module, closed at its end."""
    made = {}

    def get(shape):
        if shape not in made:
            rp, ci, va, nc = csr_of(shape)
            made[shape] = new_handle(rp, ci, va, nc)
        return made[shape]
    yield get
    for A in made.values():
        A.close()


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def nan_buffer(*shape):
    import torch
    return torch.full(shape, float("nan"), dtype=torch.float64, device="cuda")


def host(t):
    import torch
    torch.cuda.synchronize()
    return t.cpu().numpy()


def status_of(fn, *args):
    with pytest.raises(_cabi.SpmmError) as e:
        fn(*args)
    return e.value.status


# ---------------------------------------------------------------- 1. every form, many segments, against the oracle
@gpu
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("kernel", ["auto", "rows", "merge"])
def test_forms_vs_oracle(oracle, handle, shape, k, kernel):
    rp, ci, va, nc = csr_of(shape)
    A = handle(shape)
    n = A.n_rows
    B = np.random.default_rng(k).integers(1, 101, (nc, k)).astype(np.float64)
    ref = oracle.spmm(rp.astype(np.int32), ci, va, B, k)
    dB = dev(B)

    def check(got, want, what):
        assert not np.isnan(got).any(), what
        assert_close_rel(got, want, tol=REL_TOL)

    dC = nan_buffer(n, k)
    A.multiply(dB.data_ptr(), k, dC.data_ptr(), kernel)
    check(host(dC), ref, "whole")

    # strided: columns [1, 1 + k) of B (ldb = k + 3) and C (ldc = k + 2); the other columns of C stay untouched
    Bw = np.zeros((nc, k + 3))
    Bw[:, 1:1 + k] = B
    dCw = nan_buffer(n, k + 2)
    A.multiply_strided(dev(Bw).data_ptr(), k + 3, dCw.data_ptr(), k + 2, 1, k, kernel)
    cw = host(dCw)
    check(cw[:, 1:1 + k], ref, "strided")
    assert np.isnan(cw[:, 0]).all() and np.isnan(cw[:, k + 1]).all()

    d1, d2 = nan_buffer(n, k), nan_buffer(n, k)
    A.multiply_scatter(dB.data_ptr(), k, [d1.data_ptr(), d2.data_ptr()], kernel)
    check(host(d1), ref, "scatter 0")
    check(host(d2), ref, "scatter 1")

    lo, hi = A.column_span()
    dC = nan_buffer(n, k)
    A.multiply_window(dB[lo:hi + 1].data_ptr(), lo, hi - lo + 1, k, dC.data_ptr(), kernel)
    check(host(dC), ref, "window")

    rb, re = n // 5, n - n // 7
    dC = nan_buffer(max(re - rb, 1), k)
    A.multiply_rows(rb, re, dB.data_ptr(), k, dC.data_ptr(), kernel)
    check(host(dC)[:re - rb], ref[rb:re], "row range")

    for P in (3, 8):
        total = np.zeros((n, k))
        for r in range(P):
            b, e = spmm.partition_nnz(A.nnz, P, r)
            first, last = A.nnz_range_rows(b, e)
            if last < first:
                continue
            out = nan_buffer(last - first + 1, k)
            A.multiply_nnz_range(b, e, first, last, dB.data_ptr(), k, out.data_ptr(), kernel)
            total[first:last + 1] += host(out)  # partial boundary rows summed in rank order
        check(total, ref, f"non-zero ranges P={P}")

    check(A.multiply_host(B, k, kernel), ref, "host")


# ---------------------------------------------------------------- 2. the stream kernel: bit for bit as on an int32 handle
@gpu
@pytest.mark.parametrize("shape", ["fem_like", "empty_rows", "rect_tall", "cop20k_small"])
@pytest.mark.parametrize("k", [1, 2, 4, 8])
def test_stream_bitwise_as_int32_handle(handle, shape, k):
    rp, ci, va, nc = csr_of(shape)
    A = handle(shape)
    B = np.random.default_rng(k).standard_normal((nc, k))
    dB = dev(B)
    got, want = nan_buffer(A.n_rows, k), nan_buffer(A.n_rows, k)
    A.multiply(dB.data_ptr(), k, got.data_ptr(), "stream")
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp.astype(np.int32), A.n_rows, nc)) as A32:
        A32.multiply(dB.data_ptr(), k, want.data_ptr(), "stream")
    assert np.array_equal(host(got).view(np.uint64), host(want).view(np.uint64))


@gpu
def test_stream_refused_before_any_launch(handle):
    """The hub row is too long for the stream kernel: nothing is written, not even by the segments before it."""
    A = handle("hub")
    dC = nan_buffer(A.n_rows, 1)
    dB = dev(np.ones((A.n_cols, 1)))
    assert status_of(A.multiply, dB.data_ptr(), 1, dC.data_ptr(), "stream") == _cabi.SPMM_ERR_INVALID
    assert np.isnan(host(dC)).all()


# ---------------------------------------------------------------- 3. creation and queries
@gpu
@pytest.mark.parametrize("shape", list(SHAPES))
def test_queries(handle, shape):
    rp, ci, va, nc = csr_of(shape)
    A = handle(shape)
    got = A.download64()
    for g, w in zip(got, (rp, ci, va)):
        assert g.dtype == w.dtype and g.tobytes() == w.tobytes()
    lens = np.diff(rp)
    sched = A.schedule()
    hist, _ = np.histogram(lens, bins=[0, 1, 3, 5, 9, 17, 33, 257, 1 << 40])
    assert list(sched["bins"].values()) == hist.tolist()
    assert sched["max_row_len"] == lens.max()
    assert sched["mean_row_len"] == pytest.approx(len(ci) / A.n_rows)
    assert sched["auto_kernel"] == ("merge" if shape == "hub" else "rows")
    assert A.column_span() == (ci.min(), ci.max())
    nnz = len(ci)
    for b, e in [(0, nnz), (0, 1), (nnz - 1, nnz), (nnz // 3, 2 * nnz // 3), (SEG, SEG + 1), (SEG - 1, 2 * SEG + 1)]:
        if e > nnz or b >= e:
            continue
        first = np.searchsorted(rp, b, "right") - 1
        last = np.searchsorted(rp, e - 1, "right") - 1
        assert A.nnz_range_rows(b, e) == (first, last)


def raw_create_host64(n, nnz, rp, ci, va):
    h = C.c_void_p()
    return _cabi.lib().spmm_csr_create_host64(0, n, n, nnz, rp, ci, va, C.byref(h)), h


@gpu
def test_creation_checks():
    rp, ci, va, nc = csr_of("fem_like")
    n, nnz = len(rp) - 1, len(ci)
    bad0, badn = rp.copy(), rp.copy()
    bad0[0] = 1
    badn[-1] -= 1
    for args in [(bad0.ctypes.data, ci.ctypes.data, va.ctypes.data), (badn.ctypes.data, ci.ctypes.data, va.ctypes.data),
                 (None, ci.ctypes.data, va.ctypes.data), (rp.ctypes.data, None, va.ctypes.data),
                 (rp.ctypes.data, ci.ctypes.data, None)]:
        rc, h = raw_create_host64(n, nnz, *args)
        assert rc == _cabi.SPMM_ERR_INVALID and not h.value
    for bad in (bad0, badn):
        t = [dev(bad), dev(ci), dev(va)]
        for copy in (True, False):
            assert status_of(spmm.DeviceCSR.from_csr64, *t, n, nc, 0, copy) == _cabi.SPMM_ERR_INVALID
    h = C.c_void_p()
    assert _cabi.lib().spmm_csr_create_device64(0, n, n, nnz, None, None, None, 1, C.byref(h)) == _cabi.SPMM_ERR_INVALID


@gpu
def test_refusals(handle):
    rp, ci, va, nc = csr_of("fem_like")
    A = handle("fem_like")
    L, h = _cabi.lib(), A.handle
    p = C.c_void_p()
    for rc in [L.spmm_csr_build_tiles(h, -1, 0), L.spmm_csr_build_tiles_for_k(h, -1, 0, 16),
               L.spmm_csr_build_bsr(h, -1, None), L.spmm_csr_column_block(h, 0, 10, C.byref(p)),
               L.spmm_csr_device_ptrs(h, None, None, None), L.spmm_csr_download(h, None, None, None)]:
        assert rc == _cabi.SPMM_ERR_UNSUPPORTED
        assert b"64-bit" in L.spmm_last_error()
    k = 16
    dB, dC = dev(np.ones((nc, k))), nan_buffer(A.n_rows, k)
    for kernel in ("tiled", "bsr"):
        assert status_of(A.multiply, dB.data_ptr(), k, dC.data_ptr(), kernel) == _cabi.SPMM_ERR_UNSUPPORTED
        assert status_of(A.multiply_scatter, dB.data_ptr(), k, [dC.data_ptr()], kernel) == _cabi.SPMM_ERR_UNSUPPORTED
    assert np.isnan(host(dC)).all()
    assert status_of(A.download) == _cabi.SPMM_ERR_UNSUPPORTED
    assert A.tile_info()["rows_per_tile"] == 0
    # and the 64-bit queries refuse an int32 handle
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp.astype(np.int32), A.n_rows, nc)) as A32:
        assert status_of(A32.download64) == _cabi.SPMM_ERR_UNSUPPORTED
        assert L.spmm_csr_device_ptrs64(A32.handle, None, None, None) == _cabi.SPMM_ERR_UNSUPPORTED


@gpu
@pytest.mark.parametrize("source", ["host", "device_copy", "device_borrow"])
def test_from_csr64_sources(oracle, source):
    rp, ci, va, nc = csr_of("hub")
    n, k = len(rp) - 1, 8
    _cabi.tune("seg.max_nnz", SEG)
    try:
        if source == "host":
            A = spmm.DeviceCSR.from_csr64(rp, ci, va, n, nc)
        else:
            A = spmm.DeviceCSR.from_csr64(dev(rp), dev(ci), dev(va), n, nc, copy=source == "device_copy")
    finally:
        _cabi.tune("reset", 0)
    with A:
        B = np.random.default_rng(1).integers(1, 101, (nc, k)).astype(np.float64)
        dC = nan_buffer(n, k)
        A.multiply(dev(B).data_ptr(), k, dC.data_ptr())
        assert_close_rel(host(dC), oracle.spmm(rp.astype(np.int32), ci, va, B, k))
        assert all(g.tobytes() == w.tobytes() for g, w in zip(A.download64(), (rp, ci, va)))


# ---------------------------------------------------------------- 4. new values across segments
def tensor_over(ptr, n):
    import torch

    class View:
        __cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (int(ptr), False), "version": 3}
    return torch.as_tensor(View(), device="cuda")


@gpu
@pytest.mark.parametrize("kernel", ["auto", "merge"])
def test_update_values(oracle, kernel):
    rp, ci, va, nc = csr_of("hub")
    n, k, nnz = len(rp) - 1, 16, len(ci)
    B = np.random.default_rng(2).standard_normal((nc, k))
    dB = dev(B)

    def check(A, vals):
        dC = nan_buffer(n, k)
        A.multiply(dB.data_ptr(), k, dC.data_ptr(), kernel)
        assert_close_rel(host(dC), oracle.spmm(rp.astype(np.int32), ci, vals, B, k), rp, ci, vals, B)

    rng = np.random.default_rng(3)
    with new_handle(rp, ci, va, nc) as A:
        v1 = rng.standard_normal(nnz)
        A.update_values(v1)  # host form
        check(A, v1)
        v2 = rng.standard_normal(nnz)
        A.update_values(dev(v2))  # device form, another array
        check(A, v2)
        p = C.c_void_p()
        _cabi.check(_cabi.lib().spmm_csr_device_ptrs64(A.handle, None, None, C.byref(p)))
        own = tensor_over(p.value, nnz)
        own.mul_(-3.0)  # the handle's own array edited in place
        A.update_values(own)
        check(A, -3.0 * v2)
    tv = dev(va)
    _cabi.tune("seg.max_nnz", SEG)
    try:
        A = spmm.DeviceCSR.from_csr64(dev(rp), dev(ci), tv, n, nc, copy=False)
    finally:
        _cabi.tune("reset", 0)
    with A:
        tv.mul_(0.5)  # a borrowed handle: the caller's array edited in place
        A.update_values(tv)
        check(A, 0.5 * va)


# ---------------------------------------------------------------- 5. past 2^31 stored entries
BIG_N, BIG_W = 1 << 26, 33  # 2,214,592,512 non-zeros, 3 segments of at most 2^30


def big_rows_numpy(rows, k):
    """C rows of the banded matrix from its closed form: columns (r + j - 16) mod n, values 1 + ((33 r + j) mod 7) / 8;
    B[i, c] = (3 i + 5 c) mod 11 - 5. Every product and sum is exact in binary64."""
    r = np.asarray(rows, dtype=np.int64)[:, None]
    j = np.arange(BIG_W, dtype=np.int64)[None, :]
    cols = (r + j - 16) % BIG_N
    vals = 1.0 + ((BIG_W * r + j) % 7) / 8.0
    Bv = ((3 * cols[..., None] + 5 * np.arange(k)) % 11 - 5).astype(np.float64)
    return (vals[..., None] * Bv).sum(axis=1)


@gpu
def test_past_int32_offsets():
    import torch
    n, w, k = BIG_N, BIG_W, 8
    nnz = n * w
    need = nnz * 12 + 3 * n * k * 8 + (n + 1) * 12 + (6 << 30)  # A, B, C and the rank sum, row pointers, chunk temporaries
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need / 2**30:.1f} GiB free on the device, {free / 2**30:.1f} GiB are")
    rowptr = torch.arange(n + 1, dtype=torch.int64, device="cuda") * w
    colidx = torch.empty(nnz, dtype=torch.int32, device="cuda")
    vals = torch.empty(nnz, dtype=torch.float64, device="cuda")
    j = torch.arange(w, dtype=torch.int64, device="cuda")
    step = 1 << 22
    for r0 in range(0, n, step):
        r = torch.arange(r0, min(n, r0 + step), dtype=torch.int64, device="cuda")[:, None]
        colidx[r0 * w:(r0 + r.shape[0]) * w] = ((r + j - 16) % n).to(torch.int32).reshape(-1)
        vals[r0 * w:(r0 + r.shape[0]) * w] = (1.0 + ((w * r + j) % 7).to(torch.float64) / 8.0).reshape(-1)
        del r
    B = torch.empty((n, k), dtype=torch.float64, device="cuda")
    c = torch.arange(k, dtype=torch.int64, device="cuda")
    for r0 in range(0, n, step):
        i = torch.arange(r0, min(n, r0 + step), dtype=torch.int64, device="cuda")[:, None]
        B[r0:r0 + i.shape[0]] = ((3 * i + 5 * c) % 11 - 5).to(torch.float64)
    del i
    torch.cuda.empty_cache()
    A = spmm.DeviceCSR.from_csr64(rowptr, colidx, vals, n, n, copy=False)
    assert A.nnz == nnz > 2**31
    per_seg = (1 << 30) // w  # the cuts lie at most 31 rows before multiples of this (alignment step back)
    rows = set()
    for s in range(1, nnz // (1 << 30) + 1):
        rows.update(range(s * per_seg - 160, s * per_seg + 64))
    rows.update(range(0, 64))
    rows.update(range((1 << 31) // w - 64, (1 << 31) // w + 64))  # the row holding non-zero 2^31 and its neighbours
    rows.update(range(n - 64, n))
    rows.update(np.random.default_rng(0).integers(0, n, 4096).tolist())
    rows = np.array(sorted(rows))
    want = big_rows_numpy(rows, k)
    idx = torch.from_numpy(rows).cuda()
    C_auto = torch.full((n, k), float("nan"), dtype=torch.float64, device="cuda")
    other = torch.full((n, k), float("nan"), dtype=torch.float64, device="cuda")
    for kernel, dst in (("auto", C_auto), ("merge", other)):
        A.multiply(B.data_ptr(), k, dst.data_ptr(), kernel)
        torch.cuda.synchronize()
        assert np.array_equal(dst[idx].cpu().numpy(), want), kernel
    assert torch.equal(other, C_auto)
    # the 8 non-zero ranges of the non-zero strategy, the last one across 2^31, summed in rank order
    other.zero_()
    straddles = False
    for r in range(8):
        b, e = spmm.partition_nnz(nnz, 8, r)
        straddles |= b < 2**31 < e
        first, last = A.nnz_range_rows(b, e)
        assert (first, last) == (b // w, (e - 1) // w)
        out = torch.full((last - first + 1, k), float("nan"), dtype=torch.float64, device="cuda")
        A.multiply_nnz_range(b, e, first, last, B.data_ptr(), k, out.data_ptr())
        other[first:last + 1] += out
        del out
    assert straddles
    assert torch.equal(other, C_auto)
    A.close()


# ---------------------------------------------------------------- 6. without a device
def test_prototypes_cover_the_64bit_entries():
    for name in ("spmm_csr_create_host64", "spmm_csr_create_device64", "spmm_csr_device_ptrs64", "spmm_csr_download64"):
        assert name in _cabi.PROTOTYPES


@pytest.mark.parametrize("case", ["rowptr_int32", "colidx_int64", "vals_float32", "rowptr_length", "vals_length",
                                  "strided", "mixed"])
def test_from_csr64_rejects_bad_arrays_before_any_call(monkeypatch, case):
    def no_call():
        raise AssertionError("the library was called")
    monkeypatch.setattr(_cabi, "lib", no_call)
    rp = np.array([0, 2, 3, 5], dtype=np.int64)
    ci = np.array([0, 1, 2, 0, 2], dtype=np.int32)
    va = np.ones(5)
    n = 3
    if case == "rowptr_int32":
        rp = rp.astype(np.int32)
    elif case == "colidx_int64":
        ci = ci.astype(np.int64)
    elif case == "vals_float32":
        va = va.astype(np.float32)
    elif case == "rowptr_length":
        n = 4
    elif case == "vals_length":
        va = np.ones(6)
    elif case == "strided":
        va = np.ones(10)[::2]
    elif case == "mixed":
        ci = list(ci)
    with pytest.raises(ValueError):
        spmm.DeviceCSR.from_csr64(rp, ci, va, n, 3)
