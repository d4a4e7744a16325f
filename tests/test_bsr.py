"""The BSR view of a CSR handle (spmm_csr_build_bsr) and its kernel (spmm_bsr.cu, SPMM_KERNEL_BSR).

CPU tests: fem_blocked yields exactly b-blocked matrices, and a numpy restatement of the pattern rule agrees with the
generator and with every refused case. GPU tests: detection, parity against the oracle, bit identity across team shapes,
k-slabs and launch forms (the kernel runs one FMA chain per (row, column) in storage order from +0.0, as the CSR kernels
do), IEEE special values, value updates, and dispatch. Where the order of a sum does not matter the data are small
integers (A in {-2,-1,1,2}, B in [-3,3]), so results are compared bit for bit."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

from sparsematrixmultiplicationmpi_b200 import generators as gen
from conftest import REL_TOL, assert_close_rel

gpu = pytest.mark.gpu
KEEP_NAN = np.array([0x7FF80000DEADBEEF], dtype=np.uint64).view(np.float64)[0]

# k values for which AUTO takes the BSR kernel on a handle with a view (spmm_dispatch.cu, bsr_auto_k; profiles/r3_bsr.md)
def AUTO_BSR_KS(k):
    return k >= 128


# ---------------------------------------------------------------- host helpers
def csr_from_records(n_rows, rows, cols, vals):
    """The library's CSR build of general records: each row ordered by (column, value)."""
    rows, cols, vals = np.asarray(rows, np.int64), np.asarray(cols, np.int64), np.asarray(vals, np.float64)
    order = np.lexsort((vals, cols, rows))
    rp = np.concatenate(([0], np.cumsum(np.bincount(rows, minlength=n_rows)))).astype(np.int32)
    return rp, cols[order].astype(np.int32), vals[order]


def bsr_rule(rp, ci, b):
    """The pattern rule of spmm_csr_build_bsr in numpy: (True, None) or (False, first failing block row or -1)."""
    n = len(rp) - 1
    if n % b:
        return False, -1
    for R in range(n // b):
        s0, L0 = rp[R * b], rp[R * b + 1] - rp[R * b]
        if L0 % b:
            return False, R
        cq = ci[s0:s0 + L0:b].astype(np.int64)
        if (cq % b).any():
            return False, R
        want = (cq[:, None] + np.arange(b)[None, :]).reshape(-1)
        for i in range(b):
            s, L = rp[R * b + i], rp[R * b + i + 1] - rp[R * b + i]
            if L != L0 or not np.array_equal(ci[s:s + L], want):
                return False, R
    return True, None


def blocked_csr(seed, b, n_brows, n_bcols, mean_blocks, hub=None, empty_every=0, values="int"):
    """Rows of b x b blocks: block row R holds ~mean_blocks distinct block columns (sorted), hub = {R: blocks}."""
    rng = np.random.default_rng(seed)
    nb = np.minimum(rng.poisson(mean_blocks, n_brows), n_bcols)
    if empty_every:
        nb[::empty_every] = 0
    for R, m in (hub or {}).items():
        nb[R] = m
    rows, cols = [], []
    for R in range(n_brows):
        bc = np.sort(rng.choice(n_bcols, nb[R], replace=False))
        i, q, t = np.meshgrid(np.arange(b), np.arange(nb[R]), np.arange(b), indexing="ij")
        rows.append((R * b + i).reshape(-1))
        cols.append((bc[q] * b + t).reshape(-1))
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    if values == "int":
        vals = rng.choice(np.array([-2.0, -1.0, 1.0, 2.0]), rows.size)
    elif values == "normal":
        vals = rng.standard_normal(rows.size)
    else:
        vals = 0.5 + rng.random(rows.size)
    rp = np.concatenate(([0], np.cumsum(np.bincount(rows, minlength=n_brows * b)))).astype(np.int32)
    return rp, cols.astype(np.int32), vals  # rows were emitted in storage order


def broken(case, b=3):
    """A b-blocked matrix with one defect; returns (n_rows, n_cols, rp, ci, va)."""
    rp, ci, va = blocked_csr(5, b, 40, 40, 4)
    rp, ci, va = rp.astype(np.int64), ci.copy(), va.copy()
    n = len(rp) - 1
    r = 7 * b + 1  # second row of block row 7
    s, e = rp[r], rp[r + 1]
    assert e - s >= 2 * b

    def insert(pos, col, val):
        nonlocal rp, ci, va
        ci, va = np.insert(ci, pos, col), np.insert(va, pos, val)
        rp[r + 1:] += 1

    def delete(lo, hi):
        nonlocal rp, ci, va
        ci, va = np.delete(ci, np.arange(lo, hi)), np.delete(va, np.arange(lo, hi))
        rp[r + 1:] -= hi - lo

    if case == "missing":
        delete(s + 1, s + 2)
    elif case == "extra":
        insert(e, ci[e - 1] + 1 if ci[e - 1] + 1 < 40 * b else 0, 1.0)
    elif case == "duplicate":
        insert(s + 1, ci[s + 1], va[s + 1])
    elif case == "shifted":
        for i in range(b):  # the first group of every row of the block row, one column to the right
            rr = 7 * b + i
            ci[rp[rr]:rp[rr] + b] += 1
    elif case == "n_rows":
        rp = np.append(rp, rp[-1])
        n += 1
    elif case == "unequal":
        delete(s, s + b)  # a whole group: the row length stays a multiple of b
    return n, 40 * b, rp.astype(np.int32), ci.astype(np.int32), va


BROKEN = ["missing", "extra", "duplicate", "shifted", "n_rows", "unequal"]
FEM_SMALL = {b: (1500, 11_000) for b in (2, 3, 4, 5, 6)}  # node count, node-level entries


def fem_small(b, seed=3):
    nn, nz = FEM_SMALL[b]
    n, nc, r, c, v, sym = gen.fem_blocked(b, nn, nz, seed)
    assert not sym
    return n, nc, csr_from_records(n, r, c, v)


# ================================================================ CPU
@pytest.mark.parametrize("b,nodes,node_nnz", [(3, 40_397, 291_592), (4, 30_298, 164_020), (6, 20_199, 72_898)])
def test_fem_blocked_has_cfg2_size_and_is_exactly_blocked(b, nodes, node_nnz):
    n, nc, r, c, v, sym = gen.fem_blocked(b, nodes, node_nnz, 20)
    assert (n, nc, r.size, sym) == (nodes * b, nodes * b, node_nnz * b * b, False)
    assert ((0.5 <= v) & (v < 1.5)).all()
    rp, ci, _ = csr_from_records(n, r, c, v)
    assert bsr_rule(rp, ci, b) == (True, None)


@pytest.mark.parametrize("b", [2, 3, 4, 5, 6])
def test_rule_accepts_generated_blocks(b):
    n, _, (rp, ci, _) = fem_small(b)
    assert bsr_rule(rp, ci, b) == (True, None)
    rp, ci, _ = blocked_csr(b, b, 50, 60, 3, empty_every=4)
    assert bsr_rule(rp, ci, b) == (True, None)


def test_rule_follows_divisibility():
    """A 6-blocked pattern is 2- and 3-blocked; a 4-blocked one is 2-blocked, not 3-blocked."""
    rp, ci, _ = blocked_csr(1, 6, 30, 30, 3)
    assert [bsr_rule(rp, ci, b)[0] for b in (2, 3, 4, 5, 6)] == [True, True, False, False, True]
    rp, ci, _ = blocked_csr(1, 4, 30, 30, 3)
    assert [bsr_rule(rp, ci, b)[0] for b in (2, 3, 4)] == [True, False, True]


@pytest.mark.parametrize("case", BROKEN)
def test_rule_refuses_each_defect(case):
    n, nc, rp, ci, va = broken(case)
    ok, R = bsr_rule(rp, ci, 3)
    assert not ok and R in ((-1,) if case == "n_rows" else (7,))


# ================================================================ GPU
def _gpu():
    import torch
    import sparsematrixmultiplicationmpi_b200 as spmm
    from sparsematrixmultiplicationmpi_b200 import _cabi
    return torch, spmm, _cabi


def dev(a):
    torch, _, _ = _gpu()
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def cur():
    torch, _, _ = _gpu()
    return torch.cuda.current_stream().cuda_stream


def last_kernel():
    _, _, _cabi = _gpu()
    return (_cabi.lib().spmm_last_kernel_name() or b"").decode()


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def assert_bitwise(got, ref, what=""):
    got, ref = np.ascontiguousarray(got), np.ascontiguousarray(ref)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    diff = bits(got) != bits(ref)
    if diff.any():
        i = tuple(np.argwhere(diff)[0])
        raise AssertionError(f"{what}: {int(diff.sum())} entries differ, first at {i}: got {got[i]!r} want {ref[i]!r} "
                             f"(last kernel {last_kernel()})")


def assert_ieee(got, ref, what=""):
    """NaN where the reference has NaN; every other entry bit for bit (Inf by sign, 0.0 against -0.0)."""
    got, ref = np.ascontiguousarray(got), np.ascontiguousarray(ref)
    gn, rn = np.isnan(got), np.isnan(ref)
    bad = (gn != rn) | (~rn & (bits(got) != bits(ref)))
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError(f"{what}: {int(bad.sum())} entries differ, first at {i}: got {got[i]!r} want {ref[i]!r}")


def int_B(seed, n, k):
    return np.random.default_rng(seed).integers(-3, 4, (n, k)).astype(np.float64)


def nan_c(n, k, fill=np.nan):
    torch, _, _ = _gpu()
    return torch.full((n, k), fill, dtype=torch.float64, device="cuda")


def handle(rp, ci, va, n, nc):
    _, spmm, _ = _gpu()
    return spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, nc), 0)


def multiply(A, dB, k, kernel):
    torch, _, _ = _gpu()
    dC = nan_c(A.n_rows, k)
    A.multiply(dB.data_ptr(), k, dC.data_ptr(), kernel, cur())
    torch.cuda.synchronize()
    return dC.cpu().numpy()


def exact(rp, ci, va, nc, B):
    n = len(rp) - 1
    return (sp.csr_matrix((va.astype(np.int64), ci, rp), shape=(n, nc)) @ B.astype(np.int64)).astype(np.float64)


def status_of(fn):
    _, _, _cabi = _gpu()
    with pytest.raises(_cabi.SpmmError) as e:
        fn()
    return e.value.status, str(e.value)


@pytest.fixture
def tuning_reset():
    _, _, _cabi = _gpu()
    _cabi.tune("reset", 0)
    yield
    _cabi.tune("reset", 0)


# ---------------------------------------------------------------- detection
@gpu
@pytest.mark.parametrize("b", [2, 3, 4, 5, 6])
def test_each_block_size_is_accepted(b):
    n, nc, (rp, ci, va) = fem_small(b)
    with handle(rp, ci, va, n, nc) as A:
        assert A.build_bsr(b) == b
        assert A.build_bsr(-1) == max(d for d in (2, 3, 4, 5, 6) if bsr_rule(rp, ci, d)[0])


@gpu
def test_largest_block_size_is_taken():
    for b in (6, 4):
        rp, ci, va = blocked_csr(11, b, 300, 300, 5)
        n = len(rp) - 1
        with handle(rp, ci, va, n, n) as A:
            assert A.build_bsr(-1) == b  # a 6-blocked matrix is also 2- and 3-blocked, a 4-blocked one 2-blocked
            assert A.build_bsr(2) == 2


@gpu
def test_zero_drops_the_view():
    _, _, _cabi = _gpu()
    rp, ci, va = blocked_csr(12, 3, 200, 200, 4)
    n = len(rp) - 1
    with handle(rp, ci, va, n, n) as A:
        assert A.build_bsr(-1) == 3
        assert A.build_bsr(0) == 0
        st, msg = status_of(lambda: multiply(A, dev(int_B(1, n, 8)), 8, "bsr"))
        assert st == _cabi.SPMM_ERR_INVALID and "spmm_csr_build_bsr" in msg


@gpu
@pytest.mark.parametrize("case", BROKEN)
def test_each_defect_is_refused(case):
    _, _, _cabi = _gpu()
    n, nc, rp, ci, va = broken(case)
    with handle(rp, ci, va, n, nc) as A:
        st, msg = status_of(lambda: A.build_bsr(3))
        assert st == _cabi.SPMM_ERR_UNSUPPORTED
        assert ("block row 7 " in msg) if case != "n_rows" else ("not a multiple" in msg), msg
        assert A.build_bsr(-1) in (0, 2)  # the rest of the matrix may still be 2-blocked, never 3- or 6-blocked


@gpu
def test_failed_check_keeps_the_view_in_force():
    rp, ci, va = blocked_csr(13, 2, 200, 200, 4)
    n = len(rp) - 1
    with handle(rp, ci, va, n, n) as A:
        assert A.build_bsr(2) == 2
        with pytest.raises(Exception):
            A.build_bsr(4)
        B = int_B(2, n, 8)
        assert_bitwise(multiply(A, dev(B), 8, "bsr"), exact(rp, ci, va, n, B))


@gpu
@pytest.mark.parametrize("b", [1, 7, -2])
def test_bad_block_sizes_are_invalid(b):
    _, _, _cabi = _gpu()
    rp, ci, va = blocked_csr(14, 2, 20, 20, 2)
    n = len(rp) - 1
    with handle(rp, ci, va, n, n) as A:
        assert status_of(lambda: A.build_bsr(b))[0] == _cabi.SPMM_ERR_INVALID


@gpu
def test_empty_matrix_and_empty_block_rows():
    n = 12
    with handle(np.zeros(n + 1, np.int32), np.zeros(0, np.int32), np.zeros(0), n, n) as A:
        assert A.build_bsr(-1) == 6
        got = multiply(A, dev(int_B(3, n, 5)), 5, "bsr")
        assert_bitwise(got, np.zeros((n, 5)))  # +0.0 everywhere
    rp, ci, va = blocked_csr(15, 5, 300, 300, 3, empty_every=3)
    n = len(rp) - 1
    with handle(rp, ci, va, n, n) as A:
        assert A.build_bsr(5) == 5
        B = int_B(4, n, 7)
        assert_bitwise(multiply(A, dev(B), 7, "bsr"), exact(rp, ci, va, n, B))


# ---------------------------------------------------------------- parity
PARITY_KS = [1, 2, 3, 4, 7, 8, 12, 16, 32, 33, 64, 100, 128, 130, 300]


@gpu
@pytest.mark.parametrize("b", [2, 3, 4, 5, 6])
@pytest.mark.parametrize("k", PARITY_KS)
def test_bsr_vs_oracle(oracle, b, k):
    rp, ci, va = blocked_csr(20 + b, b, 2400 // b, 2400 // b, 24 // b + 1, values="pos")
    n = len(rp) - 1
    B = np.random.default_rng(b * 1000 + k).integers(1, 101, (n, k)).astype(np.float64)
    ref = oracle.spmm(rp, ci, va, B, k)
    with handle(rp, ci, va, n, n) as A:
        assert A.build_bsr(b) == b
        got = multiply(A, dev(B), k, "bsr")
        assert last_kernel() == "spmm_bsr_kernel"
    assert_close_rel(got, ref, tol=REL_TOL)


@gpu
@pytest.mark.parametrize("shape", ["hub", "empty_block_rows", "rect_wide", "rect_tall"])
@pytest.mark.parametrize("k", [5, 64])
def test_bsr_shapes_vs_oracle(oracle, shape, k):
    b = 3
    n_brows, n_bcols, kw = {"hub": (500, 2000, {"hub": {250: 1500}}), "empty_block_rows": (900, 900, {"empty_every": 2}),
                            "rect_wide": (300, 1500, {}), "rect_tall": (1500, 200, {})}[shape]
    rp, ci, va = blocked_csr(31, b, n_brows, n_bcols, 6, values="normal", **kw)
    n, nc = n_brows * b, n_bcols * b
    B = np.random.default_rng(k).standard_normal((nc, k))
    ref = oracle.spmm(rp, ci, va, B, k)
    with handle(rp, ci, va, n, nc) as A:
        assert A.build_bsr(-1) == b
        got = multiply(A, dev(B), k, "bsr")
    assert_close_rel(got, ref, rp, ci, va, B)


# ---------------------------------------------------------------- bit identity
@gpu
@pytest.mark.parametrize("b", [2, 3, 4, 5, 6])
@pytest.mark.parametrize("k", [1, 6, 17, 64, 130])
def test_integer_data_is_exact(b, k):
    rp, ci, va = blocked_csr(40 + b, b, 3000 // b, 3000 // b, 30 // b, empty_every=9)
    n = len(rp) - 1
    B = int_B(k, n, k)
    with handle(rp, ci, va, n, n) as A:
        assert A.build_bsr(b) == b
        assert_bitwise(multiply(A, dev(B), k, "bsr"), exact(rp, ci, va, n, B), f"b={b} k={k}")


SLABS = [  # (k_begin, k_count, extra columns of ldb, extra columns of ldc, B shift, C shift)
    (0, 64, 0, 0, 0, 0), (1, 33, 3, 5, 0, 0), (3, 16, 1, 0, 0, 0), (5, 7, 2, 2, 1, 0), (0, 40, 0, 0, 0, 1),
    (2, 30, 1, 3, 1, 1), (63, 1, 0, 0, 0, 0)]


@gpu
@pytest.mark.parametrize("b", [3, 4, 6])
def test_every_k_slab_equals_the_whole(b):
    """One FMA chain per (row, column): the whole multiply equals every strided slab bit for bit (odd ldb / ldc, odd
    k_begin, B or C one double off 16 bytes), and columns outside a slab keep their NaN payloads."""
    torch, _, _ = _gpu()
    rp, ci, va = blocked_csr(50 + b, b, 3000 // b, 3000 // b, 30 // b, values="normal")
    n, K = len(rp) - 1, 64
    B = np.random.default_rng(b).standard_normal((n, K))
    with handle(rp, ci, va, n, n) as A:
        assert A.build_bsr(b) == b
        whole = multiply(A, dev(B), K, "bsr")
        for k0, kc, xb, xc, sb, sc in SLABS:
            ldb, ldc = K + xb, K + xc
            bufB = torch.empty(n * ldb + 2, dtype=torch.float64, device="cuda")
            dB = bufB[sb:sb + n * ldb]
            dB.view(n, ldb)[:, :K] = dev(B)
            bufC = torch.full((n * ldc + 2,), KEEP_NAN, dtype=torch.float64, device="cuda")
            dC = bufC[sc:sc + n * ldc]
            A.multiply_strided(dB.data_ptr(), ldb, dC.data_ptr(), ldc, k0, kc, "bsr", cur())
            torch.cuda.synchronize()
            got = dC.view(n, ldc).cpu().numpy()
            what = f"slab {k0}+{kc} ldb={ldb} ldc={ldc} shifts={sb},{sc}"
            assert_bitwise(got[:, k0:k0 + kc], whole[:, k0:k0 + kc], what)
            outside = np.ones(ldc, bool)
            outside[k0:k0 + kc] = False
            assert (bits(got[:, outside]) == bits(np.float64(KEEP_NAN))).all(), what


# ---------------------------------------------------------------- IEEE special values
@gpu
@pytest.mark.parametrize("b", [2, 3, 6])
@pytest.mark.parametrize("k", [1, 5, 16])
def test_ieee_special_values(oracle, b, k):
    """0*Inf with stored +-0.0, +Inf + -Inf, NaN B rows, rows of -0.0 products (+0.0): NaN and Inf where the oracle has
    them, zeros with the oracle's signs. Integer data: every finite entry is exact, FMA or not."""
    rng = np.random.default_rng(b * 10 + k)
    rp, ci, va = blocked_csr(60 + b, b, 1200 // b, 1200 // b, 12 // b + 1, empty_every=7)
    n = len(rp) - 1
    va = va.copy()
    va[rng.random(va.size) < 0.05] = 0.0
    va[rng.random(va.size) < 0.05] = -0.0
    B = int_B(b + k, n, k)
    B[rng.choice(n, 20, replace=False)] = np.inf
    B[rng.choice(n, 20, replace=False)] = -np.inf
    B[rng.choice(n, 10, replace=False)] = np.nan
    # one block row whose every product is -0.0: its rows must come out +0.0
    R = 5
    s, e = rp[R * b], rp[R * b + b]
    if e > s:
        va[s:e] = -1.0
        for c in np.unique(ci[s:e]):
            B[c] = 0.0
    ref = oracle.spmm(rp, ci, va, B, k)
    with handle(rp, ci, va, n, n) as A:
        assert A.build_bsr(b) == b
        got = multiply(A, dev(B), k, "bsr")
    assert_ieee(got, ref, f"b={b} k={k}")
    if e > s:
        assert (bits(got[R * b:R * b + b]) == 0).all()  # +0.0


# ---------------------------------------------------------------- values
@gpu
@pytest.mark.parametrize("form", ["host", "device", "in_place"])
def test_update_values_then_bsr_equals_a_fresh_handle(form):
    torch, _, _ = _gpu()
    b, k = 3, 16
    rp, ci, va = blocked_csr(70, b, 900, 900, 8, values="normal")
    n = len(rp) - 1
    new = np.random.default_rng(71).standard_normal(va.size)
    B = np.random.default_rng(72).standard_normal((n, k))
    with handle(rp, ci, new, n, n) as F:
        assert F.build_bsr(b) == b
        want = multiply(F, dev(B), k, "bsr")
    with handle(rp, ci, va, n, n) as A:
        assert A.build_bsr(b) == b
        multiply(A, dev(B), k, "bsr")
        if form == "host":
            A.update_values(new)
        elif form == "device":
            A.update_values(dev(new), stream=cur())
        else:
            _, _, _cabi = _gpu()
            p = C.c_void_p()
            _cabi.check(_cabi.lib().spmm_csr_device_ptrs(A.handle, None, None, C.byref(p)))
            own = torch.as_tensor(type("V", (), {"__cuda_array_interface__": {
                "shape": (va.size,), "typestr": "<f8", "data": (p.value, False), "version": 3}})(), device="cuda")
            own.copy_(dev(new))
            A.update_values(own, stream=cur())
        assert_bitwise(multiply(A, dev(B), k, "bsr"), want, form)


# ---------------------------------------------------------------- dispatch
def auto_takes_bsr(k):
    return AUTO_BSR_KS(k)


@gpu
@pytest.mark.parametrize("k", [1, 2, 3, 4, 8, 16, 32, 33, 64, 128])
def test_auto_takes_bsr_inside_its_k_range(tuning_reset, k):
    b = 3
    n, nc, (rp, ci, va) = fem_small(b)
    B = np.random.default_rng(k).standard_normal((nc, k))
    with handle(rp, ci, va, n, nc) as A, handle(rp, ci, va, n, nc) as P:
        assert A.build_bsr(b) == b
        names, plain_names = [], []
        for _ in range(12):  # beyond the calls after which AUTO builds its lazy tile layout
            got = multiply(A, dev(B), k, "auto")
            names.append(last_kernel())
            plain = multiply(P, dev(B), k, "auto")
            plain_names.append(last_kernel())
            if not auto_takes_bsr(k):
                assert_bitwise(got, plain)  # the same choices as without a view
        if auto_takes_bsr(k):
            assert set(names) == {"spmm_bsr_kernel"}
            assert A.tile_info()["rows_per_tile"] == 0  # BSR launches neither count toward nor build the tile layout
            assert_bitwise(got, multiply(A, dev(B), k, "bsr"))
        else:
            assert names == plain_names and "spmm_bsr_kernel" not in names


@gpu
def test_hub_rows_stay_on_merge(tuning_reset):
    b = 3
    rp, ci, va = blocked_csr(80, b, 400, 2000, 3, hub={200: 1600}, values="normal")
    n, nc = 400 * b, 2000 * b
    B = np.random.default_rng(1).standard_normal((nc, 16))
    with handle(rp, ci, va, n, nc) as A:
        assert A.schedule()["auto_kernel"] == "merge"
        assert A.build_bsr(b) == b
        multiply(A, dev(B), 16, "auto")
        assert last_kernel() == "spmm_merge_kernel"


@gpu
def test_without_a_view_auto_is_unchanged(tuning_reset):
    b, k = 4, 32
    n, nc, (rp, ci, va) = fem_small(b)
    B = np.random.default_rng(3).standard_normal((nc, k))
    with handle(rp, ci, va, n, nc) as A, handle(rp, ci, va, n, nc) as P:
        assert A.build_bsr(b) == b and A.build_bsr(0) == 0
        for _ in range(12):
            got, name = multiply(A, dev(B), k, "auto"), last_kernel()
            want, pname = multiply(P, dev(B), k, "auto"), last_kernel()
            assert name == pname and name != "spmm_bsr_kernel"
            assert_bitwise(got, want)


@gpu
def test_partial_forms_refuse_bsr():
    torch, _, _cabi = _gpu()
    b, k = 2, 8
    rp, ci, va = blocked_csr(90, b, 200, 200, 4)
    n = len(rp) - 1
    dB, dC = dev(int_B(1, n, k)), nan_c(n, k)
    with handle(rp, ci, va, n, n) as A:
        assert A.build_bsr(b) == b
        U = _cabi.SPMM_ERR_UNSUPPORTED
        assert status_of(lambda: A.multiply_rows(0, n, dB.data_ptr(), k, dC.data_ptr(), "bsr", cur()))[0] == U
        assert status_of(lambda: A.multiply_nnz_range(0, A.nnz, 0, n - 1, dB.data_ptr(), k, dC.data_ptr(), "bsr",
                                                      cur()))[0] == U
        assert status_of(lambda: A.multiply_window(dB.data_ptr(), 0, n, k, dC.data_ptr(), "bsr", cur()))[0] == U
        assert status_of(lambda: A.multiply_scatter(dB.data_ptr(), k, [dC.data_ptr()], "bsr", cur()))[0] == U
        hB, hC = int_B(1, n, k), np.empty((n, k))
        assert status_of(lambda: _cabi.check(_cabi.lib().spmm_multiply_rows_host(
            A.handle, 0, n, hB.ctypes.data, k, hC.ctypes.data, _cabi.KERNEL_BSR)))[0] == U
    with handle(rp, ci, va, n, n) as P:
        assert status_of(lambda: multiply(P, dB, k, "bsr"))[0] == _cabi.SPMM_ERR_INVALID


@gpu
@pytest.mark.parametrize("k", [5, 64])
def test_host_forms_match_the_device_form(k):
    _, _, _cabi = _gpu()
    b = 3
    rp, ci, va = blocked_csr(91, b, 1000, 1000, 8, values="normal")
    n = len(rp) - 1
    B = np.random.default_rng(k).standard_normal((n, k))
    with handle(rp, ci, va, n, n) as A:
        assert A.build_bsr(b) == b
        want = multiply(A, dev(B), k, "bsr")
        assert_bitwise(A.multiply_host(B, k, "bsr"), want, "multiply_host")
        rows_in = [np.ascontiguousarray(B[i]) for i in range(n)]
        rows_out = [np.full(k, np.nan) for _ in range(n)]
        pin = (C.c_void_p * n)(*[r.ctypes.data for r in rows_in])
        pout = (C.c_void_p * n)(*[r.ctypes.data for r in rows_out])
        _cabi.check(_cabi.lib().spmm_multiply_host_rows(A.handle, pin, k, pout, _cabi.KERNEL_BSR))
        assert_bitwise(np.stack(rows_out), want, "multiply_host_rows")


@gpu
@pytest.mark.parametrize("k", [8, 64])
def test_six_chained_launches_without_a_host_synchronize(k):
    torch, _, _ = _gpu()
    b, steps = 4, 6
    rp, ci, va = blocked_csr(92, b, 1500, 1500, 2, empty_every=11)  # rows of <= ~28 entries: (2*28)^6*3 < 2^53
    n = len(rp) - 1
    assert np.diff(rp).max() * 2 <= 80
    X0 = int_B(k, n, k)
    xs = [X0.astype(np.int64)]
    A_int = sp.csr_matrix((va.astype(np.int64), ci, rp), shape=(n, n))
    for _ in range(steps):
        xs.append(A_int @ xs[-1])
    with handle(rp, ci, va, n, n) as A:
        assert A.build_bsr(b) == b
        multiply(A, dev(np.zeros((n, k))), k, "bsr")  # CTA cuts computed and cached before the chain
        s = torch.cuda.Stream()
        bufs = [dev(X0)] + [nan_c(n, k) for _ in range(steps)]
        s.wait_stream(torch.cuda.current_stream())
        for t in range(steps):
            A.multiply(bufs[t].data_ptr(), k, bufs[t + 1].data_ptr(), "bsr", s.cuda_stream)
        torch.cuda.synchronize()
        for t in range(1, steps + 1):
            assert_bitwise(bufs[t].cpu().numpy(), xs[t].astype(np.float64), f"step {t}")
