"""Parity of the CUDA path against the oracle, through the C-ABI (include/spmm_b200.h). B200 only."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import sparsematrixmultiplicationmpi_b200 as spmm
from sparsematrixmultiplicationmpi_b200 import _cabi, generators as gen
from conftest import GOLDEN, REL_TOL, assert_close_rel, random_csr

pytestmark = pytest.mark.gpu


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def gpu_multiply(m, B, k, kernel="auto", tune=None):
    """C = A*B through spmm_multiply_device with device-resident operands."""
    _cabi.tune("reset", 0)
    for key, val in (tune or {}).items():
        _cabi.tune(key, val)
    try:
        with spmm.DeviceCSR.from_host(m, 0) as A:
            dB = dev(B)
            dC = torch.full((m.numRows, k), np.nan, dtype=torch.float64, device="cuda")
            A.multiply(dB.data_ptr(), k, dC.data_ptr(), kernel, torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            return dC.cpu().numpy()
    finally:
        _cabi.tune("reset", 0)


# ---------------------------------------------------------------- golden vectors (reference outputs)
def test_kat_report_example(golden_multiply):
    g = golden_multiply
    m = spmm.SparseMatrix(g["kat_vals"], g["kat_colidx"], g["kat_rowptr"], 4, 4)
    for kernel in ("rows", "merge"):
        assert np.array_equal(gpu_multiply(m, g["kat_B"], 3, kernel), g["kat_C"])  # small integers: exact
    assert np.array_equal(spmm.sparseMatrixFatVectorMultiply(m, g["kat_B"], 3), g["kat_C"])


@pytest.mark.parametrize("name", ["small", "hub", "k1", "k8"])
@pytest.mark.parametrize("kernel", ["rows", "merge"])
def test_golden_cases(golden_multiply, name, kernel):
    g = golden_multiply
    rp, ci, va, B = g[f"{name}_rowptr"], g[f"{name}_colidx"], g[f"{name}_vals"], g[f"{name}_B"]
    n, k = len(rp) - 1, B.shape[1]
    got = gpu_multiply(spmm.SparseMatrix(va, ci, rp, n, n), B, k, kernel)
    assert_close_rel(got, g[f"{name}_C_seq"], rp, ci, va, B)


# ---------------------------------------------------------------- kernel families x k x shapes vs the oracle
SHAPES = {
    # name: (seed, n_rows, n_cols, mean_len, long_row, empty_every)
    "short": (1, 3000, 3000, 4, None, 9),
    "fem_like": (2, 2500, 2500, 22, None, 0),
    "hub": (3, 1200, 1200, 6, 40000, 5),
    "rect_wide": (4, 700, 5000, 12, None, 0),
    "rect_tall": (5, 5000, 300, 3, None, 4),
    "single_row": (6, 1, 64, 40, None, 0),
    "all_empty": (7, 50, 50, 0, None, 0),
}


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("k", [1, 2, 3, 4, 7, 8, 12, 16, 32, 33, 64, 100, 128, 130, 300])
@pytest.mark.parametrize("kernel", ["rows", "merge"])
def test_kernels_vs_oracle(oracle, shape, k, kernel):
    seed, n, nc, mean, long_row, empty_every = SHAPES[shape]
    if shape == "hub" and k > 64:
        pytest.skip("hub row x wide k: covered at k<=64")
    rp, ci, va = random_csr(seed, n, nc, mean, long_row=long_row, empty_every=empty_every, positive=True)
    B = np.random.default_rng(seed + k).integers(1, 101, (nc, k)).astype(np.float64)
    ref = oracle.spmm(rp, ci, va, B, k)
    got = gpu_multiply(spmm.SparseMatrix(va, ci, rp, n, nc), B, k, kernel)
    # positive data: the north_star contract verbatim, |x-ref| <= 1e-12*|ref| per entry
    assert_close_rel(got, ref, tol=REL_TOL)


@pytest.mark.parametrize("tune", [
    {"rows.kl": 32, "rows.nv": 1}, {"rows.kl": 16, "rows.nv": 2}, {"rows.kl": 8, "rows.nv": 4, "rows.unroll": 4},
    {"rows.kl": 8, "rows.nv": 4, "rows.unroll": 1}, {"rows.vec": 1}, {"rows.vec": 1, "rows.kl": 32, "rows.nv": 2},
    {"rows.ctas_per_sm": 1}, {"merge.items": 64}, {"merge.items": 4096},
])
@pytest.mark.parametrize("kernel", ["rows", "merge"])
def test_team_shape_overrides(oracle, tune, kernel):
    rp, ci, va = random_csr(11, 2000, 2000, 20, long_row=5000, empty_every=13, positive=True)
    B = np.random.default_rng(5).integers(1, 101, (2000, 64)).astype(np.float64)
    got = gpu_multiply(spmm.SparseMatrix(va, ci, rp, 2000, 2000), B, 64, kernel, tune)
    assert_close_rel(got, oracle.spmm(rp, ci, va, B, 64), tol=REL_TOL)


@pytest.mark.parametrize("k", [1, 5, 32, 64])
@pytest.mark.parametrize("tune", [{}, {"merge.wave": 4}, {"merge.wave": 64, "merge.items": 64}])
def test_merge_long_rows_only(oracle, k, tune):
    """A shard whose rows average far more than 256 non-zeros (the first non-zero range of an R-MAT matrix): the merge-path
    kernel cuts it into fewer teams, and every row is a run of many carry slots that the fix-up walks eight at a time
    (runs of 1 to ~400 slots here, with and without unused slots between them), next to a few empty rows."""
    rng = np.random.default_rng(41)
    n, nc = 40, 6000
    lens = rng.integers(300, 3000, n)
    lens[[3, 17, 18]] = 0
    lens[7] = 25000
    rp = np.concatenate(([0], np.cumsum(lens))).astype(np.int32)
    ci = np.concatenate([np.sort(rng.integers(0, nc, int(l))) for l in lens]).astype(np.int32) if rp[-1] else np.zeros(0, np.int32)
    va = 0.5 + rng.random(int(rp[-1]))
    B = rng.integers(1, 101, (nc, k)).astype(np.float64)
    got = gpu_multiply(spmm.SparseMatrix(va, ci, rp, n, nc), B, k, "merge", tune)
    assert_close_rel(got, oracle.spmm(rp, ci, va, B, k), tol=REL_TOL)


@pytest.mark.parametrize("np_", [1, 2, 4, 8, 16, 32])
@pytest.mark.parametrize("k", [1, 2, 4, 8])
def test_side_by_side_nonzeros(oracle, np_, k):
    rp, ci, va = random_csr(12, 1500, 1500, 21, long_row=700, empty_every=10, positive=True)
    B = np.random.default_rng(6).integers(1, 101, (1500, k)).astype(np.float64)
    got = gpu_multiply(spmm.SparseMatrix(va, ci, rp, 1500, 1500), B, k, "rows", {"rows.np": np_, "rows.unroll": 2})
    assert_close_rel(got, oracle.spmm(rp, ci, va, B, k), tol=REL_TOL)


# ---------------------------------------------------------------- sub-ranges used by the strategies
@pytest.mark.parametrize("kernel", ["rows", "merge"])
def test_row_blocks_and_nnz_ranges(oracle, kernel):
    n, k = 900, 16
    rp, ci, va = random_csr(14, n, n, 9, long_row=6000, empty_every=6, positive=True)
    m = spmm.SparseMatrix(va, ci, rp, n, n)
    B = np.random.default_rng(8).integers(1, 101, (n, k)).astype(np.float64)
    seq = oracle.spmm(rp, ci, va, B, k)
    dB = dev(B)
    with spmm.DeviceCSR.from_host(m, 0) as A:
        for P in (1, 3, 8):
            # a4: every rank's row block
            for r in range(P):
                s, e = spmm.partition_rows(n, P, r)
                out = torch.full((e - s, k), np.nan, dtype=torch.float64, device="cuda")
                A.multiply_rows(s, e, dB.data_ptr(), k, out.data_ptr(), kernel)
                assert_close_rel(out.cpu().numpy(), seq[s:e], tol=REL_TOL)
            # a6: every rank's non-zero range; partial boundary rows summed in rank order
            total = np.zeros((n, k))
            for r in range(P):
                b, e = spmm.partition_nnz(m.nnz, P, r)
                first, last = A.nnz_range_rows(b, e)
                assert rp[first] <= b < rp[first + 1] and rp[last] <= e - 1 < rp[last + 1]
                out = torch.full((last - first + 1, k), np.nan, dtype=torch.float64, device="cuda")
                A.multiply_nnz_range(b, e, first, last, dB.data_ptr(), k, out.data_ptr(), kernel)
                total[first:last + 1] += out.cpu().numpy()
            assert_close_rel(total, oracle.spmm(rp, ci, va, B, k, "nnz", P), tol=REL_TOL)


def test_column_slabs_strided(oracle):
    n, k = 800, 12
    rp, ci, va = random_csr(15, n, n, 10, empty_every=8, positive=True)
    B = np.random.default_rng(9).integers(1, 101, (n, k)).astype(np.float64)
    seq = oracle.spmm(rp, ci, va, B, k)
    dB = dev(B)
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, n), 0) as A:
        for P in (1, 5, 16):  # 16 > k: leading ranks own no column, the last owns all extras (ColumnWise.cpp:25-28)
            out = torch.zeros((n, k), dtype=torch.float64, device="cuda")
            for r in range(P):
                s, e = spmm.partition_cols(k, P, r)
                A.multiply_strided(dB.data_ptr(), k, out.data_ptr(), k, s, e - s)
            assert_close_rel(out.cpu().numpy(), seq, tol=REL_TOL)


def test_column_block_submatrix(oracle):
    n, k = 1000, 8
    rp, ci, va = random_csr(16, n, n, 14, empty_every=5, positive=True)
    B = np.random.default_rng(10).integers(1, 101, (n, k)).astype(np.float64)
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, n), 0) as A:
        total = np.zeros((n, k))
        nnz = 0
        for r in range(3):
            c0, c1 = spmm.partition_rows(n, 3, r)
            with A.column_block(c0, c1) as S:
                h = S.download()
                keep = (ci >= c0) & (ci < c1)
                assert np.array_equal(h.colIndices, ci[keep] - c0) and np.array_equal(h.values, va[keep])
                nnz += h.nnz
                total += S.multiply_host(B[c0:c1], k)
        assert nnz == len(ci)
        assert_close_rel(total, oracle.spmm(rp, ci, va, B, k), tol=REL_TOL)


# ---------------------------------------------------------------- CSR construction: bit-exact
LOADER = ["general_unsorted", "symmetric", "pattern", "duplicates", "skew_symmetric", "rectangular",
          "pattern_symmetric", "empty_rows", "random_symmetric"]


@pytest.mark.parametrize("name", LOADER)
def test_loader_bit_exact_vs_reference_golden(golden_loader, name):
    m = spmm.readMatrixMarketFile(os.path.join(GOLDEN, name + ".mtx"))
    g = golden_loader
    assert [m.numRows, m.numCols] == g[f"{name}_shape"].tolist()
    assert m.rowPtr.tobytes() == g[f"{name}_rowptr"].tobytes()
    assert m.colIndices.tobytes() == g[f"{name}_colidx"].tobytes()
    assert m.values.tobytes() == g[f"{name}_vals"].tobytes()


def test_device_csr_build_bit_exact_on_cop20k_shape(oracle):
    n, nc, r, c, v, sym = gen.cop20k_A_shaped()
    with spmm.DeviceCSR.from_coo_host(n, nc, r, c, v, sym) as A:
        got = A.download()
        sched = A.schedule()
    rp, ci, va = oracle.csr_from_coo(n, r, c, v, sym)
    assert got.nnz == 2624331
    assert got.rowPtr.tobytes() == rp.tobytes() and got.colIndices.tobytes() == ci.tobytes()
    assert got.values.tobytes() == va.tobytes()
    assert sum(sched["bins"].values()) == n and sched["max_row_len"] == int(np.diff(rp).max())
    assert sched["bins"]["0"] == int((np.diff(rp) == 0).sum()) and sched["auto_kernel"] == "rows"


def test_device_csr_build_ties_and_negative_zero(oracle):
    rng = np.random.default_rng(3)
    m = 20000
    r, c = rng.integers(0, 50, m), rng.integers(0, 50, m)
    v = rng.choice([-2.5, -1.0, 1.0, 1.0, 3.25, 1e-300, -1e300], m)
    with spmm.DeviceCSR.from_coo_host(50, 50, r, c, v, False) as A:
        got = A.download()
    rp, ci, va = oracle.csr_from_coo(50, r, c, v, False)
    assert got.rowPtr.tobytes() == rp.tobytes() and got.colIndices.tobytes() == ci.tobytes()
    assert got.values.tobytes() == va.tobytes()


def test_csr_build_rejects_out_of_range():
    with pytest.raises(_cabi.SpmmError):
        spmm.DeviceCSR.from_coo_host(3, 3, [0, 3], [0, 0], [1., 2.])
    with pytest.raises(_cabi.SpmmError):
        spmm.DeviceCSR.from_coo_host(2, 4, [0], [3], [1.], symmetric=True)  # mirror would leave the matrix


def test_upload_download_roundtrip_is_bitwise():
    rp, ci, va = random_csr(17, 500, 700, 8, long_row=900, empty_every=3)
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, 500, 700), 0) as A:
        h = A.download()
    assert h.rowPtr.tobytes() == rp.tobytes() and h.colIndices.tobytes() == ci.tobytes() and h.values.tobytes() == va.tobytes()


# ---------------------------------------------------------------- the reference-shaped entry points (host buffers)
def test_entry_points_single_rank(oracle):
    n, _, r, c, v, sym = gen.uniform_random(10_000, 10, seed=1)  # BASELINE.json configs[0]
    rp, ci, va = oracle.csr_from_coo(n, r, c, v, sym)
    m = spmm.SparseMatrix(va, ci, rp, n, n)
    B = spmm.generateLargeFatVector(n, 4)
    seq = oracle.spmm(rp, ci, va, B, 4)
    for fn in (spmm.sparseMatrixFatVectorMultiply, spmm.sparseMatrixFatVectorMultiplyRowWise,
               spmm.sparseMatrixFatVectorMultiplyColumnWise, spmm.sparseMatrixFatVectorMultiplyNonZeroElement):
        got = fn(m, B, 4)
        assert_close_rel(got, seq, tol=REL_TOL)
        assert spmm.areMatricesEqual(got, seq, 1e-6)  # the reference's own runtime check (main.cpp:184)
    got = spmm.sparseMatrixFatVectorMultiplyColumnWise(m, B, 4, mode="slabs")
    assert_close_rel(got, seq, tol=REL_TOL)
    got = spmm.sparseMatrixFatVectorMultiply(m, [list(row) for row in B], 4)  # vector<vector<double>> shape
    assert_close_rel(got, seq, tol=REL_TOL)
    spmm.clear_cache()


def test_entry_point_argument_errors():
    m = spmm.SparseMatrix([1.], [0], [0, 1], 1, 2)
    with pytest.raises(RuntimeError):
        spmm.sparseMatrixFatVectorMultiply(m, np.ones((1, 3)), 3)  # fat vector shorter than numCols
    with pytest.raises(RuntimeError):
        spmm.sparseMatrixFatVectorMultiply(m, np.ones((2, 3)), -1)
    assert spmm.sparseMatrixFatVectorMultiply(m, np.ones((2, 3)), 0).shape == (1, 0)


# ---------------------------------------------------------------- BASELINE.json full sizes: size-independent properties
def test_cop20k_shape_all_k_vs_oracle_and_properties(oracle):
    n, nc, r, c, v, sym = gen.cop20k_A_shaped()
    with spmm.DeviceCSR.from_coo_host(n, nc, r, c, v, sym) as A:
        host = A.download()
        for k in (1, 8, 32, 64):
            B = np.random.default_rng(k).integers(1, 101, (n, k)).astype(np.float64)
            ref = oracle.spmm(host.rowPtr, host.colIndices, host.values, B, k)
            dB = dev(B)
            for kernel in ("rows", "merge", "auto"):
                dC = torch.full((n, k), np.nan, dtype=torch.float64, device="cuda")
                A.multiply(dB.data_ptr(), k, dC.data_ptr(), kernel)
                assert_close_rel(dC.cpu().numpy(), ref, tol=REL_TOL)
        # symmetry of A (pattern and values): x^T (A y) == y^T (A x) up to rounding
        x, y = torch.rand(n, 1, dtype=torch.float64, device="cuda"), torch.rand(n, 1, dtype=torch.float64, device="cuda")
        Ax, Ay = torch.empty_like(x), torch.empty_like(y)
        A.multiply(x.data_ptr(), 1, Ax.data_ptr())
        A.multiply(y.data_ptr(), 1, Ay.data_ptr())
        assert abs(float((x * Ay).sum() - (y * Ax).sum())) <= 1e-9 * float((x * Ay).sum())


def test_auto_rebuilds_its_layouts_across_k(oracle):
    """One handle, AUTO, a sequence of k that crosses every layout boundary (8-column k-tile for k <= 8, 16-column above,
    chunks shared by 2 / 4 CTAs from k = 32 / 64, row kernels for odd k and k = 2): each result against the oracle."""
    n, nc, r, c, v, sym = gen.cop20k_A_shaped(n=30_000, nnz=600_000, nx=20, ny=25, seed=7)
    _cabi.tune("reset", 0)
    _cabi.tune("tiled.auto_after", 1)
    with spmm.DeviceCSR.from_coo_host(n, nc, r, c, v, sym) as A:
        host = A.download()
        for k in (64, 4, 2, 16, 6, 8, 128, 1, 32, 5, 64):
            B = np.random.default_rng(100 + k).integers(1, 101, (n, k)).astype(np.float64)
            ref = oracle.spmm(host.rowPtr, host.colIndices, host.values, B, k)
            dB = dev(B)
            dC = torch.full((n, k), np.nan, dtype=torch.float64, device="cuda")
            for _ in range(2):  # AUTO builds the layout when a handle comes back (a single multiply never pays for it)
                dC.fill_(np.nan)
                A.multiply(dB.data_ptr(), k, dC.data_ptr(), "auto")
                torch.cuda.synchronize()
                assert_close_rel(dC.cpu().numpy(), ref, tol=REL_TOL)
            info = A.tile_info()
            if k in (4, 6, 8, 16, 32, 64, 128):
                assert info["rows_per_tile"] > 0, (k, info)  # FEM-like rows: AUTO must have built a tile layout
    _cabi.tune("reset", 0)


def test_large_banded_vs_oracle_and_properties(oracle):
    """cfg4's family: banded, 32 per row, k=16. 2^20 rows against the ORACLE (rows / merge / auto, and a row block
    generated alone), then 2^22 rows through size-independent properties (A*1 = row sums, linearity)."""
    n, k = 1 << 20, 16
    with spmm.DeviceCSR.banded(n, 32, 4096, seed=7) as A:
        host = A.download()
        B = np.random.default_rng(16).integers(1, 101, (n, k)).astype(np.float64)
        ref = oracle.spmm(host.rowPtr, host.colIndices, host.values, B, k)
        dB = dev(B)
        for kernel in ("rows", "merge", "auto"):
            dC = torch.full((n, k), np.nan, dtype=torch.float64, device="cuda")
            A.multiply(dB.data_ptr(), k, dC.data_ptr(), kernel)
            assert_close_rel(dC.cpu().numpy(), ref, tol=REL_TOL)
        # a row block generated alone (RowWise.cpp:26-29 partition) is bit-identical to those rows of the whole matrix
        s, e = spmm.partition_rows(n, 8, 3)
        with spmm.DeviceCSR.banded(n, 32, 4096, seed=7, row_begin=s, row_end=e) as blk:
            hb = blk.download()
            assert hb.values.tobytes() == host.values[host.rowPtr[s]:host.rowPtr[e]].tobytes()
            Cb = torch.full((e - s, k), np.nan, dtype=torch.float64, device="cuda")
            blk.multiply(dB.data_ptr(), k, Cb.data_ptr())
            assert_close_rel(Cb.cpu().numpy(), ref[s:e], tol=REL_TOL)
    n = 1 << 22
    with spmm.DeviceCSR.banded(n, 32, 4096, seed=7) as A:
        ones = torch.ones((n, k), dtype=torch.float64, device="cuda")
        C1 = torch.empty((n, k), dtype=torch.float64, device="cuda")
        A.multiply(ones.data_ptr(), k, C1.data_ptr())
        vals = A.download().values.reshape(n, 32)
        rowsum = torch.from_numpy(vals).cuda().sum(dim=1, keepdim=True)
        assert torch.allclose(C1, rowsum.expand(n, k), rtol=1e-12, atol=0)  # A * ones == row sums in every column
        x = torch.randint(1, 101, (n, k), device="cuda").double()
        y = torch.randint(1, 101, (n, k), device="cuda").double()
        Cx, Cy, Cz = (torch.empty((n, k), dtype=torch.float64, device="cuda") for _ in range(3))
        z = 2 * x + y
        for src, dst in ((x, Cx), (y, Cy), (z, Cz)):
            A.multiply(src.data_ptr(), k, dst.data_ptr())
        assert torch.allclose(Cz, 2 * Cx + Cy, rtol=1e-12, atol=0)  # linearity: A(2x + y) == 2 A x + A y


@pytest.mark.parametrize("scale", [18, 20])
def test_rmat_vs_oracle(oracle, scale):
    """cfg3's family: R-MAT (0.57, 0.19, 0.19), 16 edges per vertex, duplicates kept, k=32 — merge-path, row kernel and
    AUTO against the ORACLE; the schedule must pick merge; rows come out of the device build in (column, value) order."""
    with spmm.DeviceCSR.rmat(scale, 16 << scale, seed=3) as A:
        n, k = A.n_rows, 32
        sched = A.schedule()
        assert sched["max_row_len"] > 1000 and sched["bins"]["0"] > 0 and sched["auto_kernel"] == "merge"
        host = A.download()
        assert np.all(np.diff(host.rowPtr) >= 0) and host.rowPtr[-1] == 16 << scale
        B = np.random.default_rng(scale).integers(1, 101, (n, k)).astype(np.float64)
        ref = oracle.spmm(host.rowPtr, host.colIndices, host.values, B, k)
        dB = dev(B)
        for kernel in ("merge", "rows", "auto"):
            dC = torch.full((n, k), np.nan, dtype=torch.float64, device="cuda")
            A.multiply(dB.data_ptr(), k, dC.data_ptr(), kernel)
            assert_close_rel(dC.cpu().numpy(), ref, tol=REL_TOL)
        if scale == 18:
            rows = np.repeat(np.arange(n), np.diff(host.rowPtr))
            order = np.lexsort((host.values, host.colIndices, rows))
            assert np.array_equal(order, np.arange(host.nnz))
        # cfg3 at 8 ranks: equal non-zero ranges, cut rows summed in rank order == the oracle's nnz strategy
        total = np.zeros((n, k))
        for r in range(8):
            b, e = spmm.partition_nnz(host.nnz, 8, r)
            first, last = A.nnz_range_rows(b, e)
            out = torch.full((last - first + 1, k), np.nan, dtype=torch.float64, device="cuda")
            A.multiply_nnz_range(b, e, first, last, dB.data_ptr(), k, out.data_ptr(), "auto")
            total[first:last + 1] += out.cpu().numpy()
        assert_close_rel(total, ref, tol=REL_TOL)


def test_uniform_columns_vs_oracle_and_column_blocks(oracle):
    """cfg5's family: 2^19 rows, 32 uniformly scattered columns per row, k=64 — whole matrix and the 8 column blocks
    of the column-wise strategy (partials summed in rank order) against the ORACLE."""
    n, k = 1 << 19, 64
    with spmm.DeviceCSR.banded(n, 32, n // 2, seed=11) as A:  # window = the whole row: columns anywhere
        host = A.download()
        B = np.random.default_rng(5).integers(1, 101, (n, k)).astype(np.float64)
        ref = oracle.spmm(host.rowPtr, host.colIndices, host.values, B, k)
        dB = dev(B)
        for kernel in ("rows", "merge", "auto"):
            dC = torch.full((n, k), np.nan, dtype=torch.float64, device="cuda")
            A.multiply(dB.data_ptr(), k, dC.data_ptr(), kernel)
            assert_close_rel(dC.cpu().numpy(), ref, tol=REL_TOL)
        total = torch.zeros((n, k), dtype=torch.float64, device="cuda")
        part = torch.empty((n, k), dtype=torch.float64, device="cuda")
        for r in range(8):
            c0, c1 = spmm.partition_rows(n, 8, r)
            with A.column_block(c0, c1) as S:
                S.multiply(dB[c0:c1].data_ptr(), k, part.data_ptr())
                total += part
        assert_close_rel(total.cpu().numpy(), ref, tol=REL_TOL)


def test_strategy_classes_on_one_gpu(oracle):
    rp, ci, va = random_csr(19, 3000, 3000, 15, long_row=4000, empty_every=7, positive=True)
    m = spmm.SparseMatrix(va, ci, rp, 3000, 3000)
    B = np.random.default_rng(2).integers(1, 101, (3000, 16)).astype(np.float64)
    seq = oracle.spmm(rp, ci, va, B, 16)
    eng = spmm.CudaCompute()
    dB = dev(B)
    assert_close_rel(spmm.RowWise.from_host(eng, m, 16).run(dB).cpu().numpy(), seq, tol=REL_TOL)
    blk = spmm.ColumnBlocks.from_host(eng, m, 16)
    assert_close_rel(blk.run(blk.local_B(dB)).cpu().numpy(), seq, tol=REL_TOL)
    assert_close_rel(spmm.ColumnSlabs.from_host(eng, m, 16).run(dB).cpu().numpy(), seq, tol=REL_TOL)
    assert_close_rel(spmm.NonZeroRanges.from_host(eng, m, 16).run(dB).cpu().numpy(), seq, tol=REL_TOL)


@pytest.mark.parametrize("tile", [32, 100, 4096])
@pytest.mark.parametrize("k", [1, 16, 64])
def test_round_robin_row_tiles(oracle, tile, k):
    """rows.tile: CTAs take row tiles b, b+grid, ... (the large-matrix schedule) instead of one chunk each."""
    rp, ci, va = random_csr(29, 5003, 5003, 12, long_row=777, empty_every=9, positive=True)
    B = np.random.default_rng(k).integers(1, 101, (5003, k)).astype(np.float64)
    got = gpu_multiply(spmm.SparseMatrix(va, ci, rp, 5003, 5003), B, k, "rows", {"rows.tile": tile})
    assert_close_rel(got, oracle.spmm(rp, ci, va, B, k), tol=REL_TOL)


# ---------------------------------------------------------------- row tiles with TMA-staged B rows (spmm_tiled.cu)
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


def tiled_multiply(m, B, k, T, BR, tune=None, kernel="tiled"):
    _cabi.tune("reset", 0)
    for key, val in (tune or {}).items():
        _cabi.tune(key, val)
    try:
        with spmm.DeviceCSR.from_host(m, 0) as A:
            info = A.build_tiles(T, BR)
            dB = dev(B)
            dC = torch.full((m.numRows, k), np.nan, dtype=torch.float64, device="cuda")
            A.multiply(dB.data_ptr(), k, dC.data_ptr(), kernel, torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            return dC.cpu().numpy(), info
    finally:
        _cabi.tune("reset", 0)


TILED_SHAPES = {
    # name: (n, mean_len, half_band, planes, long_row, empty_every)
    "fem3": (6000, 22, 12, (-700, 0, 700), None, 0),
    "fem_hub_empty": (5003, 18, 20, (-300, 0, 300), 900, 7),
    "narrow": (3001, 5, 3, (0,), None, 3),
    "tiny": (5, 3, 2, (0,), None, 0),
}


@pytest.mark.parametrize("shape", list(TILED_SHAPES))
@pytest.mark.parametrize("k", [2, 8, 16, 30, 32, 64, 100])
def test_tiled_kernel_vs_oracle(oracle, shape, k):
    n, mean, hb, planes, long_row, ee = TILED_SHAPES[shape]
    rp, ci, va = banded_csr(31, n, mean, hb, planes, long_row, ee)
    B = np.random.default_rng(k).integers(1, 101, (n, k)).astype(np.float64)
    got, info = tiled_multiply(spmm.SparseMatrix(va, ci, rp, n, n), B, k, -1, 0)
    assert info["rows_per_tile"] > 0 and info["reuse"] > 0
    assert_close_rel(got, oracle.spmm(rp, ci, va, B, k), tol=REL_TOL)


@pytest.mark.parametrize("T,BR", [(8, 4), (16, 16), (64, 8), (64, 32), (128, 16), (248, 16)])
@pytest.mark.parametrize("tune", [{}, {"tiled.depth": 2}, {"tiled.depth": 8}, {"tiled.thr": 1, "tiled.chunk": 3},
                                  {"tiled.thr": 100, "tiled.depth": 3}, {"tiled.ksplit": 2}, {"tiled.ksplit": 4},
                                  {"tiled.ksplit": 3, "tiled.chunk": 5}])
def test_tiled_shapes_and_teams(oracle, T, BR, tune):
    """Explicit tile heights / box heights x pipeline depth, box threshold (all boxes .. all single rows), chunk
    length, CTAs per chunk: split rows (the 900-long row: 8 segments folded by shuffles), empty rows, ragged last
    tile, window wrap-around across passes. Ragged k-tiles are covered by test_tiled_kernel_vs_oracle (k = 30, 100)."""
    n, k = 3003, 48
    rp, ci, va = banded_csr(37, n, 14, 16, (-200, 0, 200), 900, 11)
    B = np.random.default_rng(3).integers(1, 101, (n, k)).astype(np.float64)
    try:
        got, info = tiled_multiply(spmm.SparseMatrix(va, ci, rp, n, n), B, k, T, BR, tune)
    except _cabi.SpmmError as e:
        assert e.status == _cabi.SPMM_ERR_UNSUPPORTED  # this tile shape needs more shared memory than an SM has
        return
    assert info["rows_per_tile"] == T and info["box_rows"] == BR
    assert_close_rel(got, oracle.spmm(rp, ci, va, B, k), tol=REL_TOL)


@pytest.mark.parametrize("shape", list(TILED_SHAPES))
@pytest.mark.parametrize("k", [2, 6, 8])
def test_tiled_kernel_8_column_k_tile(oracle, shape, k):
    """k <= 8: the window rows are 64 bytes (k-tile of 8 columns, one 16-byte access per lane). The layout is cut for k
    as AUTO cuts it, and the tiled kernel runs with the k-tile of the layout."""
    n, mean, hb, planes, long_row, ee = TILED_SHAPES[shape]
    rp, ci, va = banded_csr(33, n, mean, hb, planes, long_row, ee)
    B = np.random.default_rng(k).integers(1, 101, (n, k)).astype(np.float64)
    ref = oracle.spmm(rp, ci, va, B, k)
    _cabi.tune("reset", 0)
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, n), 0) as A:
        info = A.build_tiles(-1, 0, k)
        if not info["rows_per_tile"]:
            pytest.skip("no tile shape fits this matrix")
        dB = dev(B)
        dC = torch.full((n, k), np.nan, dtype=torch.float64, device="cuda")
        A.multiply(dB.data_ptr(), k, dC.data_ptr(), "tiled", torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        got = dC.cpu().numpy()
        assert A.tile_info()["rows_per_tile"] > 0
        assert _cabi.lib().spmm_last_kernel_name() == b"spmm_tiled_kernel"
    assert_close_rel(got, ref, tol=REL_TOL)


@pytest.mark.parametrize("group", [1, 2, 3, 4, 6])
@pytest.mark.parametrize("k", [16, 64])
def test_tiled_walking_order_of_far_band_matrices(oracle, group, k):
    """Tiles one far band apart are walked in turn (spmm_tiled.cu: set_tile_order): any group size must give the same C."""
    n, nc, r, c, v, sym = gen.cop20k_A_shaped(n=30_000, nnz=600_000, nx=20, ny=25, seed=3)
    with spmm.DeviceCSR.from_coo_host(n, nc, r, c, v, sym, device=0) as A0:
        host = A0.download()
    B = np.random.default_rng(k).integers(1, 101, (n, k)).astype(np.float64)
    ref = oracle.spmm(host.rowPtr, host.colIndices, host.values, B, k)
    _cabi.tune("reset", 0)
    _cabi.tune("tiled.group", group)
    try:
        with spmm.DeviceCSR.from_host(host, 0) as A:
            A.build_tiles(32, 16, k)
            dB = dev(B)
            dC = torch.full((n, k), np.nan, dtype=torch.float64, device="cuda")
            A.multiply(dB.data_ptr(), k, dC.data_ptr(), "tiled", torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            got = dC.cpu().numpy()
    finally:
        _cabi.tune("reset", 0)
    assert_close_rel(got, ref, tol=REL_TOL)


def test_tiled_auto_dispatch_and_refusals(oracle):
    # scattered columns: no tile shape fits -> build succeeds with no layout, AUTO keeps the CSR kernels
    rp, ci, va = random_csr(41, 4000, 400000, 30, positive=True)
    m = spmm.SparseMatrix(va, ci, rp, 4000, 400000)
    B = np.random.default_rng(4).integers(1, 101, (400000, 16)).astype(np.float64)
    got, info = tiled_multiply(m, B, 16, -1, 0, kernel="auto")
    assert_close_rel(got, oracle.spmm(rp, ci, va, B, 16), tol=REL_TOL)
    with spmm.DeviceCSR.from_host(m, 0) as A:
        if A.build_tiles(-1)["rows_per_tile"] == 0:
            dB, dC = dev(B), torch.zeros((4000, 16), dtype=torch.float64, device="cuda")
            with pytest.raises(_cabi.SpmmError):
                A.multiply(dB.data_ptr(), 16, dC.data_ptr(), "tiled")
    # odd k: the tiled kernel refuses, AUTO falls through to the row kernels
    rp, ci, va = banded_csr(43, 2000, 20, 10)
    m = spmm.SparseMatrix(va, ci, rp, 2000, 2000)
    B = np.random.default_rng(5).integers(1, 101, (2000, 33)).astype(np.float64)
    got, info = tiled_multiply(m, B, 33, -1, 0, kernel="auto")
    assert info["rows_per_tile"] > 0
    assert_close_rel(got, oracle.spmm(rp, ci, va, B, 33), tol=REL_TOL)
    with pytest.raises(_cabi.SpmmError):
        tiled_multiply(m, B, 33, -1, 0, kernel="tiled")
    # AUTO with the layout built and k >= 16 takes the tiled kernel: same numbers as asking for it
    B = np.random.default_rng(6).integers(1, 101, (2000, 64)).astype(np.float64)
    a, _ = tiled_multiply(m, B, 64, -1, 0, kernel="auto")
    b, _ = tiled_multiply(m, B, 64, -1, 0, kernel="tiled")
    assert np.array_equal(a, b)
    assert_close_rel(a, oracle.spmm(rp, ci, va, B, 64), tol=REL_TOL)


def test_tiled_mixed_sign_duplicates_and_strided(oracle, golden_multiply):
    g = golden_multiply
    rp, ci, va, B = g["k8_rowptr"], g["k8_colidx"], g["k8_vals"], g["k8_B"]
    n = len(rp) - 1
    got, info = tiled_multiply(spmm.SparseMatrix(va, ci, rp, n, n), B, 8, 32, 16)
    assert_close_rel(got, g["k8_C_seq"], rp, ci, va, B)
    # k-slab of a wider B/C (ColumnWise.cpp:25-48): columns [16, 48) of 64 through the strided entry point
    rp, ci, va = banded_csr(47, 2500, 20, 10, (-100, 0, 100))
    m = spmm.SparseMatrix(va, ci, rp, 2500, 2500)
    B = np.random.default_rng(7).integers(1, 101, (2500, 64)).astype(np.float64)
    with spmm.DeviceCSR.from_host(m, 0) as A:
        assert A.build_tiles(-1)["rows_per_tile"] > 0
        dB, dC = dev(B), torch.zeros((2500, 64), dtype=torch.float64, device="cuda")
        _cabi.check(_cabi.lib().spmm_multiply_strided_device(A.handle, dB.data_ptr(), 64, dC.data_ptr(), 64, 16, 32,
                                                             _cabi.KERNEL_TILED, None))
        torch.cuda.synchronize()
        out = dC.cpu().numpy()
    ref = oracle.spmm(rp, ci, va, B, 64)
    assert_close_rel(out[:, 16:48], ref[:, 16:48], tol=REL_TOL)
    assert not out[:, :16].any() and not out[:, 48:].any()


# ---------------------------------------------------------------- multiply with the gather fused in (spmm_multiply_scatter_device)
# ---------------------------------------------------------------- stream kernel (spmm_stream.cu): k = 1, 2, 4, 8, bit-identical
@pytest.mark.parametrize("shape", ["short", "fem_like", "rect_wide", "rect_tall", "single_row"])
@pytest.mark.parametrize("k", [1, 2, 4, 8])
@pytest.mark.parametrize("tune", [{}, {"stream.tile": 256}, {"stream.tile": 1024}])
def test_stream_kernel_bit_identical_to_the_oracle(oracle, shape, k, tune):
    seed, n, nc, mean, long_row, empty_every = SHAPES[shape]
    rp, ci, va = random_csr(seed, n, nc, mean, long_row=long_row, empty_every=empty_every, positive=False)
    B = np.random.default_rng(seed + k).standard_normal((nc, k))
    ref = oracle.spmm(rp, ci, va, B, k)
    got = gpu_multiply(spmm.SparseMatrix(va, ci, rp, n, nc), B, k, "stream", tune)
    # product rounded, then added in ascending non-zero order: the reference's own arithmetic (-ffp-contract=off)
    assert np.array_equal(got.view(np.uint64), ref.view(np.uint64))
    auto = gpu_multiply(spmm.SparseMatrix(va, ci, rp, n, nc), B, k, "auto", {"stream.kmax": 8, "stream.min_nnz": 0})  # AUTO opted in
    assert np.array_equal(auto.view(np.uint64), ref.view(np.uint64))


def test_stream_kernel_refusals_and_strided(oracle):
    rp, ci, va = random_csr(3, 1200, 1200, 6, long_row=40000, empty_every=5, positive=True)
    m = spmm.SparseMatrix(va, ci, rp, 1200, 1200)
    B = np.ones((1200, 8))
    with pytest.raises(_cabi.SpmmError, match="stream kernel"):
        gpu_multiply(m, B, 8, "stream")  # a 40,000-entry row does not fit a tile
    rp, ci, va = random_csr(4, 900, 900, 9, positive=True)
    with pytest.raises(_cabi.SpmmError, match="stream kernel"):
        gpu_multiply(spmm.SparseMatrix(va, ci, rp, 900, 900), np.ones((900, 3)), 3, "stream")
    # a 4-column slab of a 12-column fat vector (the k-slab strategy)
    B = np.random.default_rng(1).standard_normal((900, 12))
    ref = oracle.spmm(rp, ci, va, np.ascontiguousarray(B[:, 4:8]), 4)
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, 900, 900), 0) as A:
        dB, dC = dev(B), torch.full((900, 12), np.nan, dtype=torch.float64, device="cuda")
        A.multiply_strided(dB.data_ptr(), 12, dC.data_ptr(), 12, 4, 4, "stream", torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        got = dC.cpu().numpy()
    assert np.array_equal(got[:, 4:8], ref) and np.isnan(got[:, :4]).all() and np.isnan(got[:, 8:]).all()


@pytest.mark.parametrize("kernel,k", [("rows", 5), ("rows", 64), ("merge", 32), ("tiled", 64), ("tiled", 24), ("auto", 16)])
def test_scatter_multiply_same_device(oracle, kernel, k):
    """Every destination receives the same C (on one GPU the 'peers' are three buffers of the same device)."""
    rp, ci, va = banded_csr(53, 3001, 19, 12, (-150, 0, 150), long_row=400, empty_every=9)
    m = spmm.SparseMatrix(va, ci, rp, 3001, 3001)
    B = np.random.default_rng(k).integers(1, 101, (3001, k)).astype(np.float64)
    ref = oracle.spmm(rp, ci, va, B, k)
    with spmm.DeviceCSR.from_host(m, 0) as A:
        if kernel == "tiled":
            assert A.build_tiles(-1)["rows_per_tile"] > 0
        dB = dev(B)
        outs = [torch.full((3001, k), np.nan, dtype=torch.float64, device="cuda") for _ in range(3)]
        A.multiply_scatter(dB.data_ptr(), k, [o.data_ptr() for o in outs], kernel, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        for o in outs:
            assert_close_rel(o.cpu().numpy(), ref, tol=REL_TOL)
        assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
        with pytest.raises(_cabi.SpmmError):
            A.multiply_scatter(dB.data_ptr(), k, [o.data_ptr() for o in outs] * 3, kernel)  # 9 destinations


def test_rowwise_p2p_two_gpus():
    """RowWise with the gather / all-gather fused into the multiply over NVLink peer stores (needs 2 GPUs)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import subprocess
    import sys
    script = os.path.join(os.path.dirname(os.path.abspath(__file__)), "multi_gpu_p2p.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533", script],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "p2p ok" in r.stdout


@pytest.mark.parametrize("slabs", [0, 1, 2, 4])
def test_host_multiply_k_slab_pipeline(oracle, slabs):
    """spmm_multiply_host with the k-slab PCIe pipeline (host.slabs): same C as the single-shot path and the oracle."""
    n, k = 40_000, 64  # 2 x 20 MB: above the size from which AUTO pipelines
    rp, ci, va = banded_csr(59, n, 9, 30, (-500, 0, 500))
    m = spmm.SparseMatrix(va, ci, rp, n, n)
    B = np.random.default_rng(8).integers(1, 101, (n, k)).astype(np.float64)
    ref = oracle.spmm(rp, ci, va, B, k)
    _cabi.tune("reset", 0)
    _cabi.tune("host.slabs", slabs)
    try:
        with spmm.DeviceCSR.from_host(m, 0) as A:
            got = A.multiply_host(B, k, "auto")
            assert_close_rel(got, ref, tol=REL_TOL)
            again = A.multiply_host(B, k, "rows")
            assert_close_rel(again, ref, tol=REL_TOL)
    finally:
        _cabi.tune("reset", 0)


@pytest.mark.parametrize("shape", ["banded", "random", "rect_wide", "rect_tall", "mostly_empty"])
@pytest.mark.parametrize("pinned", [False, True])
def test_host_multiply_rows_and_flat_buffers(oracle, shape, pinned):
    """spmm_multiply_host (flat buffer: pinned goes straight to the copy engine, pageable through the pinned staging and
    the host threads) and spmm_multiply_host_rows (one pointer per row: the memory shape of a FatVector) give the oracle's C."""
    k = 64
    if shape == "banded":
        n, nc = 40_000, 40_000
        rp, ci, va = banded_csr(61, n, 9, 30, (-700, 0, 700))
    else:
        n, nc, mean, ee = {"random": (30_000, 30_000, 8, 0), "rect_wide": (9_000, 50_000, 10, 0),
                           "rect_tall": (50_000, 700, 3, 4), "mostly_empty": (30_000, 30_000, 1, 2)}[shape]
        rp, ci, va = random_csr(17, n, nc, mean, empty_every=ee, positive=True)
    m = spmm.SparseMatrix(va, ci, rp, n, nc)
    B = np.random.default_rng(9).integers(1, 101, (nc, k)).astype(np.float64)
    ref = oracle.spmm(rp, ci, va, B, k)
    with spmm.DeviceCSR.from_host(m, 0) as A:
        if pinned:
            Bp = torch.from_numpy(B).pin_memory()
            Cp = torch.empty((n, k), dtype=torch.float64).pin_memory()
            got = A.multiply_host(Bp.numpy(), k, "auto", Cp.numpy())
        else:
            got = A.multiply_host(B, k, "auto")
        assert_close_rel(got, ref, tol=REL_TOL)
        # FatVector shape: every row its own allocation
        rows_in = [np.ascontiguousarray(B[i]) for i in range(nc)]
        rows_out = [np.full(k, np.nan) for _ in range(n)]
        pin = (C.c_void_p * nc)(*[r.ctypes.data for r in rows_in])
        pout = (C.c_void_p * n)(*[r.ctypes.data for r in rows_out])
        _cabi.check(_cabi.lib().spmm_multiply_host_rows(A.handle, pin, k, pout, _cabi.KERNEL_AUTO))
        assert_close_rel(np.stack(rows_out), ref, tol=REL_TOL)


def test_window_multiply_reads_only_the_rows_it_is_given(oracle):
    """spmm_multiply_window_device: a row block of a banded matrix with only its own rows of B plus the halo resident."""
    n, k = 20_000, 16
    rp, ci, va = banded_csr(67, n, 12, 40, (-300, 0, 300))
    m = spmm.SparseMatrix(va, ci, rp, n, n)
    B = np.random.default_rng(2).integers(1, 101, (n, k)).astype(np.float64)
    ref = oracle.spmm(rp, ci, va, B, k)
    for P, r in ((4, 0), (4, 2), (4, 3), (1, 0)):
        s, e = spmm.partition_rows(n, P, r)
        with spmm.DeviceCSR.from_host(m.row_block(s, e), 0) as A:
            lo, hi = A.column_span()
            assert lo == ci[rp[s]:rp[e]].min() and hi == ci[rp[s]:rp[e]].max()
            window = dev(B[lo:hi + 1])  # nothing else of B exists on the device
            out = torch.full((e - s, k), np.nan, dtype=torch.float64, device="cuda")
            for kernel in ("rows", "merge", "auto"):
                A.multiply_window(window.data_ptr(), lo, hi - lo + 1, k, out.data_ptr(), kernel,
                                  torch.cuda.current_stream().cuda_stream)
                torch.cuda.synchronize()
                assert_close_rel(out.cpu().numpy(), ref[s:e], tol=REL_TOL)


def test_reduce_blocks_rank_order():
    """spmm_reduce_blocks_device: sources added in list order (the column-block strategy's reduce over peer buffers)."""
    g = torch.Generator(device="cuda").manual_seed(3)
    srcs = [torch.randn(100_002, dtype=torch.float64, device="cuda", generator=g) * 10.0 ** (3 * i) for i in range(5)]
    out = torch.empty_like(srcs[0])
    _cabi.reduce_blocks(0, [t.data_ptr() for t in srcs], out.numel(), out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    want = srcs[0].clone()
    for t in srcs[1:]:
        want += t  # ((s0 + s1) + s2) + ...
    assert torch.equal(out, want)
    with pytest.raises(_cabi.SpmmError):
        _cabi.reduce_blocks(0, [t.data_ptr() for t in srcs], 7, out.data_ptr())  # odd element count


def test_device_init_one_gpu(oracle):
    """spmm_device_init: the start-up work of a process that was given ONE GPU (context, staging arena, one tiny multiply per
    kernel module) — idempotent, refuses a device that does not exist, and leaves the library usable."""
    lib = _cabi.lib()
    assert lib.spmm_device_init(0) == 0
    assert lib.spmm_device_init(0) == 0
    assert lib.spmm_device_init(4096) != 0 and b"no such device" in lib.spmm_last_error()
    rp, ci, va = random_csr(51, 300, 300, 7, long_row=150, empty_every=11, positive=True)
    B = np.random.default_rng(2).integers(1, 101, (300, 6)).astype(np.float64)
    got = spmm.sparseMatrixFatVectorMultiply(spmm.SparseMatrix(va, ci, rp, 300, 300), B, 6)
    assert_close_rel(got, oracle.spmm(rp, ci, va, B, 6), tol=REL_TOL)
