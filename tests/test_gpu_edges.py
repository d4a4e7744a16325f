"""Parity at the edges real callers reach and the rest of the suite does not: tile layouts on rectangular and offset handles
(row blocks, column blocks, wide and tall matrices), strided / odd / misaligned operands, IEEE special values, chains of
launches on one stream without a host synchronisation, one handle on two streams, and a C of more than 2^31 elements.

Where the order of a sum does not matter the data are small integers (A in {-2,-1,1,2}, B in [-3,3]): every partial sum is
an integer below 2^53, so any order and any FMA give the same bits and the kernels are compared bit for bit with the
oracle. Tolerances are used only where rounding is the point (the bound against sum |a*b| of conftest.assert_close_rel).
C is filled with NaN before a launch, and columns a launch must not touch with a NaN of a payload of its own."""
import ctypes as C
import re

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import sparsematrixmultiplicationmpi_b200 as spmm
from sparsematrixmultiplicationmpi_b200 import _cabi
from conftest import assert_close_rel

pytestmark = pytest.mark.gpu

# a NaN no arithmetic produces (payload 0xdeadbeef): the value of C columns a launch must leave alone
KEEP_NAN = np.array([0x7FF80000DEADBEEF], dtype=np.uint64).view(np.float64)[0]


# ---------------------------------------------------------------- helpers
def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def cur():
    return torch.cuda.current_stream().cuda_stream


def last_kernel():
    return (_cabi.lib().spmm_last_kernel_name() or b"").decode()


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


@pytest.fixture
def tuning_reset():
    _cabi.tune("reset", 0)
    yield
    _cabi.tune("reset", 0)


def fem_csr(seed, n_rows, mean_len, half_band, planes=(0,), n_cols=None, hubs=None, empty_every=0, values="int",
            scattered_hubs=False):
    """FEM-like rows: the columns of row i cluster in windows of +-half_band around i * n_cols / n_rows + p for each plane
    offset p (a square matrix: around the diagonal and the next grid planes; n_cols = 3 n_rows: around 3i; n_rows = 3 n_cols:
    around i/3). hubs: {row: length} long rows, in the band like the others (repeated columns) or, with scattered_hubs, with
    columns anywhere (one staged B row per non-zero: no tile shape fits such a row, the builder then leaves the CSR kernels in
    charge; used where only the CSR kernels run). values: "int" = {-2,-1,1,2}, "normal", or "pos" [0.5, 1.5)."""
    n_cols = n_rows if n_cols is None else n_cols
    rng = np.random.default_rng(seed)
    lens = rng.poisson(mean_len, n_rows)
    if empty_every:
        lens[::empty_every] = 0
    for r, length in (hubs or {}).items():
        lens[r] = length
    rowptr = np.concatenate(([0], np.cumsum(lens))).astype(np.int32)
    rows = np.repeat(np.arange(n_rows, dtype=np.int64), lens)
    centre = rows * n_cols // n_rows + rng.choice(np.asarray(planes), rows.size)
    col = np.clip(centre + rng.integers(-half_band, half_band + 1, rows.size), 0, n_cols - 1)
    for r in (hubs or {}) if scattered_hubs else ():
        col[rowptr[r]:rowptr[r + 1]] = rng.integers(0, n_cols, lens[r])
    col = col[np.lexsort((col, rows))].astype(np.int32)
    nnz = int(rowptr[-1])
    if values == "int":
        vals = rng.choice(np.array([-2.0, -1.0, 1.0, 2.0]), nnz)
    elif values == "normal":
        vals = rng.standard_normal(nnz)
    else:
        vals = 0.5 + rng.random(nnz)
    return rowptr, col, vals


def int_B(seed, n, k):
    return np.random.default_rng(seed).integers(-3, 4, (n, k)).astype(np.float64)


def assert_bitwise(got, ref, what=""):
    got, ref = np.ascontiguousarray(got), np.ascontiguousarray(ref)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    diff = bits(got) != bits(ref)
    if diff.any():
        i = tuple(np.argwhere(diff)[0])
        raise AssertionError(f"{what}: {int(diff.sum())} entries differ, first at {i}: got {got[i]!r} want {ref[i]!r} "
                             f"(last kernel {last_kernel()})")


def assert_ieee(got, ref, what=""):
    """NaN where the reference has NaN (any payload); every other entry bit for bit (so Inf by sign and 0.0 against -0.0)."""
    got, ref = np.ascontiguousarray(got), np.ascontiguousarray(ref)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    gn, rn = np.isnan(got), np.isnan(ref)
    bad = (gn != rn) | (~rn & (bits(got) != bits(ref)))
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError(f"{what}: {int(bad.sum())} entries differ, first at {i}: got {got[i]!r} want {ref[i]!r} "
                             f"(last kernel {last_kernel()})")


def nan_c(n, k, fill=np.nan):
    return torch.full((n, k), fill, dtype=torch.float64, device="cuda")


def multiply(A, dB, k, kernel):
    dC = nan_c(A.n_rows, k)
    A.multiply(dB.data_ptr(), k, dC.data_ptr(), kernel, cur())
    torch.cuda.synchronize()
    return dC.cpu().numpy()


def shifted(n_elems, shift):
    """A float64 view of n_elems elements whose data_ptr() is `shift` doubles past a 256-byte aligned allocation."""
    buf = torch.empty(n_elems + 2, dtype=torch.float64, device="cuda")
    return buf[shift:shift + n_elems]


def device_view(ptr, n, typestr, dtype):
    """A CUDA tensor over memory the library owns (no copy)."""
    class View:
        __cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (int(ptr), False), "version": 3}
    return torch.as_tensor(View(), device="cuda").view(dtype)


# ================================================================ A. tile layouts on rectangular and offset handles
FEM_N = 120_000
FEM_KS = (4, 8, 16, 24, 64)


@pytest.fixture(scope="module")
def fem120k(oracle):
    """Three grid planes 2400 rows apart, about 22 non-zeros per row (2.6 M); integer data; the oracle's C for each k."""
    rp, ci, va = fem_csr(101, FEM_N, 22, 12, planes=(-2400, 0, 2400))
    m = spmm.SparseMatrix(va, ci, rp, FEM_N, FEM_N)
    Bs = {k: int_B(200 + k, FEM_N, k) for k in FEM_KS}
    refs = {k: oracle.spmm(rp, ci, va, Bs[k], k) for k in FEM_KS}
    return m, Bs, refs


ROW_BLOCKS = sorted({(P, r) for P in (2, 3, 8) for r in (0, P // 2, P - 1)})


@pytest.mark.parametrize("P,r", ROW_BLOCKS)
def test_tiled_row_block_handles(fem120k, tuning_reset, monkeypatch, capfd, record_property, P, r):
    """The (e-s) x n handle of one rank of the row-wise strategy: its band sits at column offset s, so the B tensor map, the
    boxes and the far-band detection see n_cols != n_rows and a band far from the local diagonal."""
    m, Bs, refs = fem120k
    s, e = spmm.partition_rows(FEM_N, P, r)
    blk = m.row_block(s, e)
    monkeypatch.setenv("SPMM_TILED_DEBUG", "1")  # the builder reports the walking order (far band, group) on stderr
    with spmm.DeviceCSR.from_host(blk, 0) as A:
        for T, BR in ((-1, 0), (32, 16)):
            for k in FEM_KS:
                info = A.build_tiles(T, BR, k)
                assert info["rows_per_tile"] > 0, (T, BR, k, info)
                got = multiply(A, dev(Bs[k]), k, "tiled")
                assert last_kernel() == "spmm_tiled_kernel"
                assert_bitwise(got, refs[k][s:e], f"rows [{s},{e}) T={T} BR={BR} k={k}")
                if r >= 1:
                    order = re.findall(r"final .*band=(-?\d+) group=(-?\d+)", capfd.readouterr().err)
                    record_property(f"T{T}_BR{BR}_k{k}", {"tile_info": info, "far_band_group": order[-1:] or None})
    # AUTO builds the layout itself on such a handle (after tiled.auto_after whole-matrix multiplies) and uses it
    _cabi.tune("tiled.auto_after", 1)
    with spmm.DeviceCSR.from_host(blk, 0) as A:
        dB = dev(Bs[16])
        first = multiply(A, dB, 16, "auto")
        again = multiply(A, dB, 16, "auto")
        assert last_kernel() == "spmm_tiled_kernel", A.tile_info()
        assert_bitwise(first, refs[16][s:e], "AUTO before the layout")
        assert_bitwise(again, refs[16][s:e], "AUTO with its layout")


@pytest.mark.parametrize("P", [3, 8])
@pytest.mark.parametrize("k", [8, 16, 64])
def test_tiled_column_block_handles(oracle, fem120k, P, k):
    """The n x w handle of one rank of the column-block strategy (local column ids), each with its own tile layout; the
    rank-order sum of the partial products is the oracle's sequential C."""
    m, Bs, refs = fem120k
    B = Bs[16] if k == 16 else int_B(300 + k, FEM_N, k)
    ref = refs[16] if k == 16 else oracle.spmm(m.rowPtr, m.colIndices, m.values, B, k)
    dB = dev(B)
    total = np.zeros((FEM_N, k))
    with spmm.DeviceCSR.from_host(m, 0) as A:
        for r in range(P):
            c0, c1 = spmm.partition_rows(FEM_N, P, r)
            with A.column_block(c0, c1) as S:
                h = S.download()
                info = S.build_tiles(-1, 0, k)
                assert info["rows_per_tile"] > 0, (r, info)
                got = multiply(S, dB[c0:c1], k, "tiled")
                assert last_kernel() == "spmm_tiled_kernel"
                assert_bitwise(got, oracle.spmm(h.rowPtr, h.colIndices, h.values, B[c0:c1], k), f"column block {r}")
                total += got
    assert_bitwise(total, ref, "rank-order sum")


@pytest.mark.parametrize("shape", ["wide", "tall"])
@pytest.mark.parametrize("k", [8, 16, 64])
def test_tiled_wide_and_tall(oracle, shape, k):
    """n x 3n with columns around 3i, and 3n x n with columns around i/3."""
    n = 20_000
    n_rows, n_cols = (n, 3 * n) if shape == "wide" else (3 * n, n)
    rp, ci, va = fem_csr(400 + k, n_rows, 22, 12, n_cols=n_cols)
    B = int_B(k, n_cols, k)
    ref = oracle.spmm(rp, ci, va, B, k)
    dB = dev(B)
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n_rows, n_cols), 0) as A:
        for T, BR in ((-1, 0), (32, 16)):
            info = A.build_tiles(T, BR, k)
            assert info["rows_per_tile"] > 0, (T, BR, info)
            got = multiply(A, dB, k, "tiled")
            assert last_kernel() == "spmm_tiled_kernel"
            assert_bitwise(got, ref, f"{shape} T={T} BR={BR}")


# ================================================================ B. strided, misaligned and scattered operands
def edge_matrix(seed=7, n=3001, hub=300, scattered_hubs=False):
    """FEM-like with a hub row and empty rows; integer data."""
    return fem_csr(seed, n, 14, 10, planes=(-250, 0, 250), hubs={n // 2: hub}, empty_every=11, scattered_hubs=scattered_hubs)


def ld(least, odd, extra):
    v = least + extra
    return v + 1 if (v % 2 == 1) != odd else v


# (k_begin, ldb odd, ldc odd): ldb != ldc in every case
STRIDE_CASES = [(1, True, False), (2, False, True), (3, False, False), (2, False, False), (0, False, False)]


def strided_expect(kernel, kc, kb, ldb, ldc):
    """None when the launch must run, else the status it must refuse with (B and C are 256-byte aligned allocations, so
    column k_begin is 16-byte aligned exactly when k_begin is even)."""
    if kernel == "tiled" and not (kc % 2 == 0 and kb % 2 == 0 and ldb % 2 == 0 and ldc % 2 == 0):
        return _cabi.SPMM_ERR_UNSUPPORTED
    if kernel == "stream" and kc >= 2 and (kb % 2 or ldb % 2):
        return _cabi.SPMM_ERR_INVALID
    return None


def _strided_case(oracle, kernel, kc):
    n = 3001
    rp, ci, va = edge_matrix()
    m = spmm.SparseMatrix(va, ci, rp, n, n)
    with spmm.DeviceCSR.from_host(m, 0) as A:
        if kernel in ("tiled", "auto"):
            assert A.build_tiles(-1, 0, max(kc, 2))["rows_per_tile"] > 0
        for kb, bodd, codd in STRIDE_CASES:
            ldb, ldc = ld(kb + kc, bodd, 0), ld(kb + kc, codd, 4)
            B = int_B(kb * 1000 + kc, n, ldb)
            ref = oracle.spmm(rp, ci, va, B[:, kb:kb + kc], kc)
            want = np.full((n, ldc), KEEP_NAN)
            want[:, kb:kb + kc] = np.nan
            dB, dC = dev(B), dev(want)
            case = f"{kernel} k_begin={kb} k_count={kc} ldb={ldb} ldc={ldc}"
            status = strided_expect(kernel, kc, kb, ldb, ldc)
            if status is not None:
                with pytest.raises(_cabi.SpmmError) as e:
                    A.multiply_strided(dB.data_ptr(), ldb, dC.data_ptr(), ldc, kb, kc, kernel, cur())
                assert e.value.status == status, case
                torch.cuda.synchronize()
                assert_bitwise(dC.cpu().numpy(), want, case + " (refused: C untouched)")
                continue
            A.multiply_strided(dB.data_ptr(), ldb, dC.data_ptr(), ldc, kb, kc, kernel, cur())
            torch.cuda.synchronize()
            got = dC.cpu().numpy()
            assert_bitwise(got[:, kb:kb + kc], ref, case)
            want[:, kb:kb + kc] = ref
            assert_bitwise(got, want, case + " (columns outside the slab)")


@pytest.mark.parametrize("kernel", ["rows", "merge", "auto", "tiled"])
@pytest.mark.parametrize("kc", [2, 16, 17, 33, 64, 65, 129])
def test_strided_odd_leading_dimensions_and_offsets(oracle, tuning_reset, kernel, kc):
    """ldb != ldc, each odd in turn, k_begin odd and even, k_count across the team widths of pick_shape."""
    _strided_case(oracle, kernel, kc)


@pytest.mark.parametrize("kc", [1, 2, 4, 8])
def test_strided_stream_kernel(oracle, tuning_reset, kc):
    _strided_case(oracle, "stream", kc)


@pytest.mark.parametrize("kernel,k", [(kn, k) for kn in ("rows", "merge", "auto", "tiled") for k in (2, 8, 16, 64)] +
                         [("stream", k) for k in (1, 2, 4, 8)])
def test_misaligned_operands(oracle, tuning_reset, kernel, k):
    """B and/or C one double past a 16-byte boundary with even k: the CSR kernels fall back to 8-byte accesses, the tiled
    kernel refuses (AUTO then takes the CSR kernels), the stream kernel refuses a misaligned B from k = 2."""
    n = 3001
    rp, ci, va = edge_matrix()
    B = int_B(k, n, k)
    ref = oracle.spmm(rp, ci, va, B, k)
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, n), 0) as A:
        if kernel in ("tiled", "auto"):
            assert A.build_tiles(-1, 0, k)["rows_per_tile"] > 0
        for b_shift, c_shift in ((1, 0), (0, 1), (1, 1)):
            dB = shifted(n * k, b_shift)
            dB.copy_(dev(B).reshape(-1))
            dC = shifted(n * k, c_shift)
            dC.fill_(np.nan)
            case = f"{kernel} k={k} B+{b_shift} C+{c_shift}"
            refuse = (kernel == "tiled" and _cabi.SPMM_ERR_UNSUPPORTED) or \
                     (kernel == "stream" and k >= 2 and b_shift and _cabi.SPMM_ERR_INVALID)
            if refuse:
                with pytest.raises(_cabi.SpmmError) as e:
                    A.multiply(dB.data_ptr(), k, dC.data_ptr(), kernel, cur())
                assert e.value.status == refuse, case
                torch.cuda.synchronize()
                assert np.isnan(dC.cpu().numpy()).all(), case
                continue
            A.multiply(dB.data_ptr(), k, dC.data_ptr(), kernel, cur())
            torch.cuda.synchronize()
            assert last_kernel() != "spmm_tiled_kernel", case
            assert_bitwise(dC.cpu().numpy().reshape(n, k), ref, case)


@pytest.mark.parametrize("kernel", ["rows", "merge", "auto", "tiled"])
@pytest.mark.parametrize("k", [5, 16])
def test_scatter_to_misaligned_destinations(oracle, tuning_reset, kernel, k):
    """Three destinations congruent modulo 16 bytes, each 8 bytes past a 16-byte boundary."""
    n = 3001
    rp, ci, va = edge_matrix()
    B = int_B(50 + k, n, k)
    ref = oracle.spmm(rp, ci, va, B, k)
    step = n * k + (n * k) % 2 + 2
    buf = torch.full((3 * step + 2,), np.nan, dtype=torch.float64, device="cuda")
    outs = [buf[1 + i * step:1 + i * step + n * k] for i in range(3)]
    assert all(o.data_ptr() % 16 == 8 for o in outs)
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, n), 0) as A:
        if kernel in ("tiled", "auto"):
            assert A.build_tiles(-1, 0, k if k % 2 == 0 else 16)["rows_per_tile"] > 0
        dB = dev(B)
        if kernel == "tiled":
            with pytest.raises(_cabi.SpmmError) as e:
                A.multiply_scatter(dB.data_ptr(), k, [o.data_ptr() for o in outs], kernel, cur())
            assert e.value.status == _cabi.SPMM_ERR_UNSUPPORTED
            torch.cuda.synchronize()
            assert torch.isnan(buf).all()
            return
        A.multiply_scatter(dB.data_ptr(), k, [o.data_ptr() for o in outs], kernel, cur())
        torch.cuda.synchronize()
    for i, o in enumerate(outs):
        assert_bitwise(o.cpu().numpy().reshape(n, k), ref, f"destination {i}")
    host = buf.cpu().numpy()
    gaps = np.concatenate([host[:1]] + [host[1 + i * step + n * k:1 + (i + 1) * step] for i in range(3)])
    assert np.isnan(gaps).all()  # nothing stored between the destinations


@pytest.mark.parametrize("kernel", ["rows", "merge"])
@pytest.mark.parametrize("k", [5, 33])
def test_row_blocks_and_nnz_ranges_into_misaligned_c(oracle, kernel, k):
    """multiply_rows / multiply_nnz_range with odd k, C 8 bytes past a 16-byte boundary, a hub row and empty rows."""
    n = 3001
    rp, ci, va = edge_matrix(hub=5000, scattered_hubs=True)
    m = spmm.SparseMatrix(va, ci, rp, n, n)
    B = int_B(k, n, k)
    ref = oracle.spmm(rp, ci, va, B, k)
    dB = dev(B)
    with spmm.DeviceCSR.from_host(m, 0) as A:
        for r in range(3):
            s, e = spmm.partition_rows(n, 3, r)
            out = shifted((e - s) * k, 1)
            out.fill_(np.nan)
            A.multiply_rows(s, e, dB.data_ptr(), k, out.data_ptr(), kernel, cur())
            torch.cuda.synchronize()
            assert_bitwise(out.cpu().numpy().reshape(e - s, k), ref[s:e], f"rows [{s},{e})")
        for r in range(8):
            b, e = spmm.partition_nnz(m.nnz, 8, r)
            first, last = A.nnz_range_rows(b, e)
            out = shifted((last - first + 1) * k, 1)
            out.fill_(np.nan)
            A.multiply_nnz_range(b, e, first, last, dB.data_ptr(), k, out.data_ptr(), kernel, cur())
            torch.cuda.synchronize()
            sub_rp = np.clip(rp[first:last + 2], b, e) - b
            want = oracle.spmm(sub_rp, ci[b:e], va[b:e], B, k)
            assert_bitwise(out.cpu().numpy().reshape(-1, k), want, f"non-zeros [{b},{e})")


# ================================================================ C. IEEE special values
def nnz_range_outputs(A, rp, dB, k, kernel, P=8):
    """[(first, last, b, e, C rows)] of every rank's non-zero range."""
    outs = []
    for r in range(P):
        b, e = spmm.partition_nnz(int(rp[-1]), P, r)
        first, last = A.nnz_range_rows(b, e)
        out = nan_c(last - first + 1, k)
        A.multiply_nnz_range(b, e, first, last, dB.data_ptr(), k, out.data_ptr(), kernel, cur())
        outs.append((first, last, b, e, out))
    torch.cuda.synchronize()
    return [(f, l, b, e, o.cpu().numpy()) for f, l, b, e, o in outs]


LEAK_RUNS = [("rows", None, (5, 8, 64)), ("merge", None, (5, 8, 64)), ("merge", {"merge.items": 64}, (5, 16)),
             ("tiled", (8, 4), (8, 16, 64)), ("tiled", (248, 16), (8, 16, 64)), ("stream", None, (1, 2, 4, 8)),
             ("nnz_rows", None, (5, 16)), ("nnz_merge", None, (5, 16))]


@pytest.mark.parametrize("kind,opt,ks", LEAK_RUNS, ids=[f"{r[0]}-{r[1]}" for r in LEAK_RUNS])
def test_loads_that_must_not_be_accumulated(oracle, tuning_reset, kind, opt, ks):
    """NaN in B row 0, in the last B row and in B rows that no non-zero names but that sit inside a staged TMA box. Rows
    that name column 0 or the last column are NaN in every column; every other row is bit for bit the result of the same
    launch with those B rows set to 0.0 (a clamped, padded or batched load that is accumulated shows as a NaN there)."""
    n = 3000
    rp, ci, va = fem_csr(77, n, 14, 10, planes=(-250, 0, 250), hubs={n // 2: 350}, empty_every=13, values="normal")
    unused = [n // 3 + 1, n // 2 + 7]
    for u in unused:
        ci[ci == u] = u + 1  # keeps every row sorted; u-1 and u+1 are still named, so u lies inside their boxes
    bad_cols = [0, n - 1] + unused
    poisoned_nz = np.isin(ci, [0, n - 1])
    rows_of = np.repeat(np.arange(n), np.diff(rp))
    R = np.unique(rows_of[poisoned_nz])
    assert (ci == 0).any() and (ci == n - 1).any() and not np.isin(ci, unused).any()
    if isinstance(opt, dict):
        for key, val in opt.items():
            _cabi.tune(key, val)
    ran = 0
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, n), 0) as A:
        for k in ks:
            if kind == "tiled":
                try:
                    assert A.build_tiles(opt[0], opt[1], k)["rows_per_tile"] == opt[0]
                except _cabi.SpmmError as e:
                    assert e.status == _cabi.SPMM_ERR_UNSUPPORTED  # this tile shape needs more shared memory than an SM has
                    continue
            ran += 1
            B = np.random.default_rng(k).standard_normal((n, k))
            Bn, Bz = B.copy(), B.copy()
            Bn[bad_cols] = np.nan
            Bz[bad_cols] = 0.0
            if kind.startswith("nnz_"):
                kern = kind[4:]
                with_nan = nnz_range_outputs(A, rp, dev(Bn), k, kern)
                with_zero = nnz_range_outputs(A, rp, dev(Bz), k, kern)
                for (f, l, b, e, cn), (_, _, _, _, cz) in zip(with_nan, with_zero):
                    hit = np.unique(rows_of[b:e][poisoned_nz[b:e]]) - f
                    clean = np.setdiff1d(np.arange(l - f + 1), hit)
                    assert np.isnan(cn[hit]).all(), (k, b, e)
                    assert not np.isnan(cz).any(), (k, b, e)
                    assert_bitwise(cn[clean], cz[clean], f"{kind} k={k} non-zeros [{b},{e})")
                continue
            kernel = kind
            cn = multiply(A, dev(Bn), k, kernel)
            cz = multiply(A, dev(Bz), k, kernel)
            assert last_kernel() == f"spmm_{kernel}_kernel"
            clean = np.setdiff1d(np.arange(n), R)
            assert np.isnan(cn[R]).all(), (kind, k)
            assert not np.isnan(cz).any(), (kind, k)
            assert_bitwise(cn[clean], cz[clean], f"{kind} {opt} k={k}")
            assert_close_rel(cz, oracle.spmm(rp, ci, va, Bz, k), rp, ci, va, Bz)
    assert ran > 0


# special B rows: +Inf, -Inf, +0.0, -0.0 in every column
C_PINF, C_NINF, C_ZERO, C_NZERO = 1000, 1001, 1002, 1003


def special_matrix(n=3000):
    """Integer FEM-like rows that never name the special B rows, then rows built to hit each IEEE case, two hub rows
    (1500 entries: cut by many merge teams) and empty rows. Returns the CSR and {case: rows}."""
    rp, ci, va = fem_csr(91, n, 14, 10, planes=(-250, 0, 250), empty_every=17)
    ci[(ci >= C_PINF) & (ci <= C_NZERO)] = C_PINF - 1  # monotone: rows stay sorted
    rows = [(ci[rp[i]:rp[i + 1]], va[rp[i]:rp[i + 1]]) for i in range(n)]
    h = 1500
    hub_cols = np.sort(np.random.default_rng(5).integers(0, C_PINF - 1, h))
    design = {
        "nan": {
            100: ([998, C_PINF, 1010], [1.0, 0.0, 2.0]),         # stored +0.0 x +Inf
            1700: ([C_NINF, 1005], [-0.0, 1.0]),                 # stored -0.0 x -Inf
            1701: ([990, C_PINF, C_NINF], [1.0, 2.0, 1.0]),      # +Inf + -Inf
            2200: (np.sort(np.r_[hub_cols[:-2], C_PINF, C_NINF]), np.r_[np.ones(h - 2), 1.0, 1.0]),  # hub: both signs
        },
        "pinf": {
            1702: ([C_PINF, C_NINF, 1007], [2.0, -1.0, 3.0]),     # +Inf reached from both B signs, one product sign
            2300: (np.sort(np.r_[hub_cols[:-1], C_PINF]), np.r_[-np.ones(h - 1), 2.0]),  # hub with one +Inf product
        },
        "ninf": {1703: ([C_PINF, 1008], [-1.0, 2.0])},
        "pzero": {
            1704: ([], []),                                       # empty
            1705: ([C_ZERO, C_NZERO, C_NZERO], [-1.0, 2.0, 1.0]),  # products -0.0, -0.0, -0.0
            1706: ([995, 996], [-0.0, -0.0]),                     # stored -0.0 x integers
            2400: (np.r_[np.full(h // 2, C_ZERO), np.full(h // 2, C_NZERO)], np.r_[-np.ones(h // 2), np.ones(h // 2)]),
        },
    }
    for case in design.values():
        for r, (c, v) in case.items():
            rows[r] = (np.asarray(c, dtype=np.int32), np.asarray(v, dtype=np.float64))
    lens = np.array([len(c) for c, _ in rows])
    rp = np.concatenate(([0], np.cumsum(lens))).astype(np.int32)
    ci = np.concatenate([c for c, _ in rows]).astype(np.int32)
    va = np.concatenate([v for _, v in rows]).astype(np.float64)
    return rp, ci, va, {case: sorted(d) for case, d in design.items()}


def special_B(n, k, seed=3):
    B = int_B(seed, n, k)
    B[C_PINF], B[C_NINF], B[C_ZERO], B[C_NZERO] = np.inf, -np.inf, 0.0, -0.0
    return B


IEEE_RUNS = [("rows", None, (1, 5, 16, 64)), ("merge", None, (1, 5, 16, 64)), ("merge", {"merge.items": 64}, (1, 5, 16, 64)),
             ("tiled", None, (8, 16, 64)), ("stream", None, (1, 2)), ("auto", None, (16, 64)),
             ("nnz_rows", None, (5, 16)), ("nnz_merge", None, (5, 16)), ("nnz_merge", {"merge.items": 64}, (5, 16))]


@pytest.mark.parametrize("kind,tune,ks", IEEE_RUNS, ids=[f"{r[0]}-{r[1]}" for r in IEEE_RUNS])
def test_ieee_special_values_propagate(oracle, tuning_reset, kind, tune, ks):
    """0 x Inf (stored +0.0 and -0.0), +Inf + -Inf -> NaN; +Inf of one sign -> +Inf; empty rows and rows of -0.0 products
    -> +0.0 (sign bit clear), also where a hub row is cut by many merge teams and inside a non-zero range."""
    n = 3000
    rp, ci, va, cases = special_matrix(n)
    for key, val in (tune or {}).items():
        _cabi.tune(key, val)
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, n), 0) as A:
        if kind in ("tiled", "auto"):
            assert A.build_tiles(-1, 0, 16)["rows_per_tile"] > 0
        for k in ks:
            B = special_B(n, k)
            ref = oracle.spmm(rp, ci, va, B, k)
            assert np.isnan(ref[cases["nan"]]).all() and (ref[cases["pinf"]] == np.inf).all()
            assert (ref[cases["ninf"]] == -np.inf).all()
            assert (bits(ref[cases["pzero"]]) == 0).all()
            dB = dev(B)
            if kind.startswith("nnz_"):
                for f, l, b, e, got in nnz_range_outputs(A, rp, dB, k, kind[4:]):
                    sub_rp = np.clip(rp[f:l + 2], b, e) - b
                    assert_ieee(got, oracle.spmm(sub_rp, ci[b:e], va[b:e], B, k), f"{kind} k={k} non-zeros [{b},{e})")
                continue
            got = multiply(A, dB, k, kind)
            if kind != "auto":
                assert last_kernel() == f"spmm_{kind}_kernel"
            assert_ieee(got, ref, f"{kind} {tune} k={k}")


@pytest.mark.parametrize("k", [5, 16])
def test_merge_carry_slots_of_an_earlier_nan_multiply(tuning_reset, k):
    """A merge multiply whose B is all NaN leaves NaN in the handle's carry slots; the next one must not read them."""
    _cabi.tune("merge.items", 64)
    n = 3000
    rp, ci, va = fem_csr(13, n, 14, 10, hubs={700: 2000, 1900: 900}, empty_every=7, scattered_hubs=True)
    m = spmm.SparseMatrix(va, ci, rp, n, n)
    B = int_B(k, n, k)
    with spmm.DeviceCSR.from_host(m, 0) as A, spmm.DeviceCSR.from_host(m, 0) as F:
        assert np.isnan(multiply(A, dev(np.full((n, k), np.nan)), k, "merge")[np.diff(rp) > 0]).all()
        again = multiply(A, dev(B), k, "merge")
        fresh = multiply(F, dev(B), k, "merge")
    assert_bitwise(again, fresh, "after a NaN multiply")


def wide_range(rng, size, lo, hi):
    return rng.choice([-1.0, 1.0], size) * (1.0 + rng.random(size)) * np.exp2(rng.integers(lo, hi + 1, size).astype(np.float64))


@pytest.mark.parametrize("k", [1, 2, 4, 8])
def test_stream_kernel_bit_identity_under_stress(oracle, tuning_reset, k):
    """Products that overflow to +-Inf, subnormal products, exact cancellation to 0, magnitudes 2^-1000 .. 2^1000: the
    stream kernel rounds each product and adds in non-zero order, as the oracle does, so the bits agree (NaN as NaN)."""
    n = 4000
    rng = np.random.default_rng(k)
    rp, ci, va = fem_csr(17 + k, n, 10, 40, empty_every=9, values="normal")
    e = rng.choice([-1, 0, 1], ci.size, p=[0.3, 0.4, 0.3])
    va = wide_range(rng, ci.size, -20, 20) * np.exp2(e * rng.integers(500, 1001, ci.size).astype(np.float64))
    # exact cancellation: in every third row the second non-zero is the first one negated, on the same column
    for i in range(0, n, 3):
        a, b = rp[i], rp[i + 1]
        if b - a >= 2:
            ci[a + 1], va[a + 1] = ci[a], -va[a]
    B = wide_range(rng, (n, k), -20, 20) * np.exp2(rng.choice([-1, 0, 1], (n, k)) * rng.integers(500, 1001, (n, k)))
    with np.errstate(over="ignore", under="ignore"):
        prods = va[:, None] * B[ci]
    assert np.isinf(prods).any() and ((prods != 0) & (np.abs(prods) < np.finfo(np.float64).tiny)).any()
    ref = oracle.spmm(rp, ci, va, B, k)
    m = spmm.SparseMatrix(va, ci, rp, n, n)
    with spmm.DeviceCSR.from_host(m, 0) as A:
        assert_ieee(multiply(A, dev(B), k, "stream"), ref, f"stream k={k}")
        _cabi.tune("stream.kmax", 8)
        _cabi.tune("stream.min_nnz", 0)
        got = multiply(A, dev(B), k, "auto")
        assert last_kernel() == "spmm_stream_kernel"
        assert_ieee(got, ref, f"AUTO -> stream k={k}")


@pytest.mark.parametrize("kernel", ["rows", "merge", "tiled", "auto"])
@pytest.mark.parametrize("k", [8, 16, 64])
def test_mixed_signs_over_a_wide_range(oracle, tuning_reset, kernel, k):
    """Random signs, |a| and |b| in 2^[-40, 40]: entries cancel, so the error is bounded against sum |a*b|."""
    n = 6000
    rng = np.random.default_rng(k)
    rp, ci, va = fem_csr(23, n, 22, 12, planes=(-700, 0, 700), hubs={n // 3: 900}, empty_every=19)
    va = wide_range(rng, ci.size, -40, 40)
    B = wide_range(rng, (n, k), -40, 40)
    ref = oracle.spmm(rp, ci, va, B, k)
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, n), 0) as A:
        if kernel in ("tiled", "auto"):
            assert A.build_tiles(-1, 0, k)["rows_per_tile"] > 0
        got = multiply(A, dev(B), k, kernel)
        if kernel != "auto":
            assert last_kernel() == f"spmm_{kernel}_kernel"
    assert_close_rel(got, ref, rp, ci, va, B)


# ================================================================ D. chains of launches on one stream
CHAIN_STEPS = 6


def chain_matrix():
    """Integer rows of at most ~40 non-zeros: (2 * 40)^6 * 3 < 2^53, so six products stay exact."""
    n = 20_000
    rp, ci, va = fem_csr(61, n, 14, 10, planes=(-400, 0, 400), empty_every=23)
    assert np.diff(rp).max() <= 40
    return n, rp, ci, va


def int_chain(rp, ci, vals_per_step, X0):
    """x_{t+1} = A_t x_t in int64 (exact)."""
    n = len(rp) - 1
    xs = [X0.astype(np.int64)]
    for v in vals_per_step:
        A = sp.csr_matrix((v.astype(np.int64), ci, rp), shape=(n, n))
        xs.append(A @ xs[-1])
    return xs


def run_chain(A, X0, k, kernels, mode, values=None):
    """Enqueue the chain on one side stream with no host synchronisation inside; returns [(step, tensor)] of kept steps."""
    s = torch.cuda.Stream()
    if mode == "raw":
        bufs = [X0] + [nan_c(A.n_rows, k) for _ in range(CHAIN_STEPS)]
    else:
        bufs = [X0.clone(), nan_c(A.n_rows, k)]
    s.wait_stream(torch.cuda.current_stream())
    for t in range(CHAIN_STEPS):
        if values is not None:
            A.update_values(values[t], stream=s.cuda_stream)
        src, dst = (bufs[t], bufs[t + 1]) if mode == "raw" else (bufs[t % 2], bufs[(t + 1) % 2])
        A.multiply(src.data_ptr(), k, dst.data_ptr(), kernels[t], s.cuda_stream)
    torch.cuda.synchronize()
    if mode == "raw":
        return list(enumerate(bufs))[1:]
    return [(CHAIN_STEPS - 1, bufs[(CHAIN_STEPS - 1) % 2]), (CHAIN_STEPS, bufs[CHAIN_STEPS % 2])]


def warm(A, k, kernels):
    """First launches compute and cache CTA cuts (with a synchronisation) and grow the merge scratch: done before a chain."""
    x, y = torch.zeros((A.n_cols, k), dtype=torch.float64, device="cuda"), nan_c(A.n_rows, k)
    for kern in set(kernels):
        A.multiply(x.data_ptr(), k, y.data_ptr(), kern, cur())
    torch.cuda.synchronize()


CHAINS = [(kn, k) for kn in ("rows", "merge", "tiled", "auto") for k in (8, 64)] + [("stream", 8)]


@pytest.mark.parametrize("mode", ["raw", "war"])
@pytest.mark.parametrize("kernel,k", CHAINS)
def test_chained_launches(tuning_reset, mode, kernel, k):
    """raw: separate buffers, each launch reads the C of the one before; war: two buffers ping-ponged, each launch also
    writes the B of the one before."""
    n, rp, ci, va = chain_matrix()
    X0 = int_B(k, n, k)
    ref = int_chain(rp, ci, [va] * CHAIN_STEPS, X0)
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, n), 0) as A:
        if kernel in ("tiled", "auto"):
            assert A.build_tiles(-1, 0, k)["rows_per_tile"] > 0
        kernels = [kernel] * CHAIN_STEPS
        warm(A, k, kernels)
        for t, x in run_chain(A, dev(X0), k, kernels, mode):
            assert_bitwise(x.cpu().numpy(), ref[t].astype(np.float64), f"{mode} {kernel} step {t}")


@pytest.mark.parametrize("mode", ["raw", "war"])
def test_chained_launches_of_mixed_kernels(tuning_reset, mode):
    n, rp, ci, va = chain_matrix()
    k = 8
    X0 = int_B(1, n, k)
    ref = int_chain(rp, ci, [va] * CHAIN_STEPS, X0)
    kernels = ["tiled", "rows", "merge", "stream", "auto", "tiled"]
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, n), 0) as A:
        assert A.build_tiles(-1, 0, k)["rows_per_tile"] > 0
        warm(A, k, kernels)
        for t, x in run_chain(A, dev(X0), k, kernels, mode):
            assert_bitwise(x.cpu().numpy(), ref[t].astype(np.float64), f"{mode} mixed step {t}")


@pytest.mark.parametrize("kernel", ["rows", "merge", "tiled", "mixed"])
def test_chained_launches_with_value_updates(tuning_reset, kernel):
    """update_values (device form, on the chain's stream) before every step: step t multiplies with values t."""
    n, rp, ci, va = chain_matrix()
    k = 8
    X0 = int_B(2, n, k)
    vals = [np.random.default_rng(100 + t).choice(np.array([-2.0, -1.0, 1.0, 2.0]), va.size) for t in range(CHAIN_STEPS)]
    ref = int_chain(rp, ci, vals, X0)
    kernels = ["tiled", "rows", "merge", "stream", "auto", "tiled"] if kernel == "mixed" else [kernel] * CHAIN_STEPS
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, n), 0) as A:
        assert A.build_tiles(-1, 0, k)["rows_per_tile"] > 0
        warm(A, k, kernels)
        dvals = [dev(v) for v in vals]
        torch.cuda.synchronize()
        for t, x in run_chain(A, dev(X0), k, kernels, "raw", dvals):
            assert_bitwise(x.cpu().numpy(), ref[t].astype(np.float64), f"{kernel} with updates, step {t}")


# ================================================================ E. one handle, two streams
def test_one_handle_two_streams_merge(oracle, tuning_reset):
    """Two whole-matrix merge multiplies of one hub-heavy handle (same k, different B) enqueued back to back on two streams:
    they share the handle's carry slots, which the library orders between the streams."""
    n, k = 200_000, 16
    hubs = {int(r): 20_000 for r in np.random.default_rng(1).choice(n, 40, replace=False)}
    rp, ci, va = fem_csr(31, n, 6, 200, hubs=hubs, empty_every=5, scattered_hubs=True)
    B1, B2 = int_B(1, n, k), int_B(2, n, k)
    refs = [oracle.spmm(rp, ci, va, B, k) for B in (B1, B2)]
    _cabi.tune("merge.items", 64)
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, n), 0) as A:
        dBs = [dev(B1), dev(B2)]
        dCs = [nan_c(n, k), nan_c(n, k)]
        streams = [torch.cuda.Stream(), torch.cuda.Stream()]
        for s in streams:
            s.wait_stream(torch.cuda.current_stream())
        for s, dB, dC in zip(streams, dBs, dCs):
            A.multiply(dB.data_ptr(), k, dC.data_ptr(), "merge", s.cuda_stream)
        torch.cuda.synchronize()
        for i, (dC, ref) in enumerate(zip(dCs, refs)):
            assert_bitwise(dC.cpu().numpy(), ref, f"stream {i}")


# ================================================================ F. a C of more than 2^31 elements
def test_c_beyond_2_31_elements(tuning_reset):
    """2^24 + 3 banded rows x k = 130: B and C hold 2.2e9 elements (17.5 GB each). A seeded sample of rows (first and last
    included) against a float64 reference of those rows, for the row, merge and tiled kernels."""
    n, k = (1 << 24) + 3, 130
    assert n * k > 2 ** 31
    free, _ = torch.cuda.mem_get_info()
    if free < (48 << 30):
        pytest.skip(f"needs 48 GB of free device memory, {free >> 30} GB free")
    with spmm.DeviceCSR.banded(n, 16, 4096, seed=5) as A:
        prow, pcol, pval = C.c_void_p(), C.c_void_p(), C.c_void_p()
        _cabi.check(_cabi.lib().spmm_csr_device_ptrs(A.handle, C.byref(prow), C.byref(pcol), C.byref(pval)))
        d_rp = device_view(prow.value, n + 1, "<i4", torch.int32)
        d_ci = device_view(pcol.value, A.nnz, "<i4", torch.int32)
        d_va = device_view(pval.value, A.nnz, "<f8", torch.float64)
        rows = np.unique(np.r_[0, n - 1, np.random.default_rng(9).choice(n, 4094, replace=False)])
        lo = d_rp[torch.from_numpy(rows).cuda()].cpu().numpy().astype(np.int64)
        hi = d_rp[torch.from_numpy(rows + 1).cuda()].cpu().numpy().astype(np.int64)
        idx = np.concatenate([np.arange(a, b) for a, b in zip(lo, hi)])
        g = torch.Generator(device="cuda").manual_seed(11)
        dB = torch.empty((n, k), dtype=torch.float64, device="cuda").random_(-3, 4, generator=g)
        cols = d_ci[torch.from_numpy(idx).cuda()].long()
        vals = d_va[torch.from_numpy(idx).cuda()].cpu().numpy()
        Bg = dB[cols].cpu().numpy()
        prods = vals[:, None] * Bg
        starts = np.r_[0, np.cumsum(hi - lo)[:-1]]
        ref, absref = np.add.reduceat(prods, starts), np.add.reduceat(np.abs(prods), starts)
        info = A.build_tiles(-1, 0, k)
        assert info["rows_per_tile"] > 0, info
        dC = torch.empty((n, k), dtype=torch.float64, device="cuda")
        sample = torch.from_numpy(rows).cuda()
        for kernel in ("rows", "merge", "tiled"):
            dC.fill_(np.nan)
            A.multiply(dB.data_ptr(), k, dC.data_ptr(), kernel, cur())
            torch.cuda.synchronize()
            assert last_kernel() == f"spmm_{kernel}_kernel"
            got = dC[sample].cpu().numpy()
            err = np.abs(got - ref)
            bad = ~(err <= 1e-12 * absref)
            assert not bad.any(), (kernel, rows[np.argwhere(bad)[0][0]], got[bad][:4], ref[bad][:4])
        del dB, dC
