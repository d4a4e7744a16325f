"""Which kernel each device multiply form runs for each kernel id, and which ids it refuses (DESIGN.md section 4.3).

Every form (spmm_multiply_device, _strided_device, _scatter_device, _window_device, _rows_device, _nnz_range_device) is
called with the ids 0 (AUTO), 1 (ROWS), 2 (MERGE), 6 (TILED), 8 (STREAM), 9 (BSR) and the unknown ids 3 and 42, on handles
that make AUTO take each of its branches: a FEM-like matrix with and without a tile layout, one with a hub row (the
schedule picks merge-path), a b = 3 blocked matrix with a BSR view, and the FEM-like matrix at k = 1 with the stream kernel
allowed. A call that succeeds must report the expected kernel and give the oracle's C bit for bit (integer data: every
partial sum is exact); a refused call must return the expected status and leave C untouched. The lazy tile layout's
counter of AUTO calls is covered on its own."""
import ctypes as C

import numpy as np
import pytest

from conftest import random_csr

pytestmark = pytest.mark.gpu

AUTO, ROWS, MERGE, TILED, STREAM, BSR = 0, 1, 2, 6, 8, 9
IDS = (AUTO, ROWS, MERGE, TILED, STREAM, BSR, 3, 42)
OK, INVALID, UNSUPPORTED = 0, 1, 4
NAME = {ROWS: "spmm_rows_kernel", MERGE: "spmm_merge_kernel", TILED: "spmm_tiled_kernel",
        STREAM: "spmm_stream_kernel", BSR: "spmm_bsr_kernel"}

# form -> what it serves: the whole matrix (device, strided), the scatter and window forms, or a part of the matrix
FORMS = {"multiply": "whole", "strided": "whole", "scatter": "scatter", "window": "window",
         "rows": "part", "rows_inner": "part", "nnz": "part", "nnz_inner": "part"}


def _gpu():
    import torch
    import sparsematrixmultiplicationmpi_b200 as spmm
    from sparsematrixmultiplicationmpi_b200 import _cabi
    return torch, spmm, _cabi


@pytest.fixture
def tuning_reset():
    _, _, _cabi = _gpu()
    _cabi.tune("reset", 0)
    yield
    _cabi.tune("reset", 0)


def int_vals(seed, n):
    return np.random.default_rng(seed).choice(np.array([-2.0, -1.0, 1.0, 2.0]), n)


def int_B(seed, n, k):
    return np.random.default_rng(seed).integers(-3, 4, (n, k)).astype(np.float64)


def csr_of_records(n, nc, r, c, v, sym):
    """The CSR the library assembles from coordinate records (integer values)."""
    _, spmm, _ = _gpu()
    with spmm.DeviceCSR.from_coo_host(n, nc, r, c, int_vals(11, len(v)), sym, device=0) as A:
        m = A.download()
    return m.rowPtr, m.colIndices, m.values, n, nc


_MATS = {}


def matrix(name):
    """(rowptr, colidx, vals, n_rows, n_cols) of one of the test matrices, generated once per session."""
    if name not in _MATS:
        from sparsematrixmultiplicationmpi_b200 import generators as gen
        if name == "fem":
            _MATS[name] = csr_of_records(*gen.cop20k_A_shaped(n=30_000, nnz=600_000, nx=20, ny=25, seed=7))
        elif name == "hub":
            rp, ci, _ = random_csr(5, 20_000, 20_000, 8, long_row=20_000)
            _MATS[name] = rp, ci, int_vals(12, int(rp[-1])), 20_000, 20_000
        else:
            _MATS[name] = csr_of_records(*gen.fem_blocked(3, 1500, 11_000, seed=3))
    return _MATS[name]


class Case:
    """A handle and a k. layout: build_tiles(-1, 0, build_k) first; stream: tune("stream.min_nnz", 1)."""

    def __init__(self, mat, k, layout=False, build_k=None, bsr=False, stream=False):
        self.mat, self.k, self.layout, self.build_k, self.bsr, self.stream = mat, k, layout, build_k or k, bsr, stream
        self.merge = mat == "hub"
        # B and C are contiguous torch allocations (16-byte aligned): the tiled kernel fits any even k, the stream kernel
        # k = 1, 2, 4, 8 (the test matrices have short rows)
        self.tiled_fits = layout and k % 2 == 0
        self.stream_fits = k in (1, 2, 4, 8)


CASES = {
    "fem": Case("fem", 16),
    "fem_tiled": Case("fem", 16, layout=True),
    "fem_tiled_odd_k": Case("fem", 15, layout=True, build_k=16),
    "hub": Case("hub", 16),
    "blocked_k64": Case("blocked", 64, bsr=True),
    "blocked_k128": Case("blocked", 128, bsr=True),
    "stream": Case("fem", 1, stream=True),
}


def expected(c, form, kid):
    """(status, kernel run): the table of DESIGN.md section 4.3, for a call that has work to do."""
    kind = FORMS[form]
    if kind == "part":
        if kid == BSR:
            return UNSUPPORTED, None
        if kid == AUTO:
            return OK, MERGE if c.merge else ROWS
        return OK, MERGE if kid == MERGE else ROWS
    if kid == BSR and kind != "whole":
        return UNSUPPORTED, None
    accepted = {"whole": (AUTO, ROWS, MERGE, TILED, STREAM, BSR), "scatter": (AUTO, ROWS, MERGE, TILED),
                "window": (AUTO, ROWS, MERGE)}[kind]
    if kid not in accepted:
        return INVALID, None
    if kid in (ROWS, MERGE):
        return OK, kid
    if kid == TILED:
        if not c.layout:
            return INVALID, None
        return (OK, TILED) if c.tiled_fits else (UNSUPPORTED, None)
    if kid == STREAM:
        return (OK, STREAM) if c.stream_fits else (INVALID, None)
    if kid == BSR:
        return (OK, BSR) if c.bsr else (INVALID, None)
    if c.merge:
        return OK, MERGE
    if kind == "whole" and c.stream and c.stream_fits:
        return OK, STREAM
    if kind == "whole" and c.bsr and c.k >= 128:
        return OK, BSR
    if kind != "window" and c.tiled_fits:  # the gate passes on the FEM-like matrix at k = 16
        return OK, TILED
    return OK, ROWS


def open_handle(c):
    _, spmm, _cabi = _gpu()
    rp, ci, va, n, nc = matrix(c.mat)
    A = spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, nc), 0)
    if c.layout:
        assert A.build_tiles(-1, 0, c.build_k)["rows_per_tile"] > 0
    if c.bsr:
        assert A.build_bsr(3) == 3
    if c.stream:
        _cabi.tune("stream.min_nnz", 1)
    return A


def call(A, form, dB, k, kid):
    """Run one form with a raw kernel id into a NaN-filled C.
    -> (status, C as numpy, the matrix rows C holds, the non-zero range multiplied)"""
    torch, _, _cabi = _gpu()
    L, h, s = _cabi.lib(), A.handle, torch.cuda.current_stream().cuda_stream
    n, nnz = A.n_rows, A.nnz
    rows = slice(0, n)
    if form in ("nnz", "nnz_inner"):
        z0, z1 = (0, nnz) if form == "nnz" else (nnz // 3, 2 * nnz // 3)
        f, l = A.nnz_range_rows(z0, z1)
        rows = slice(f, l + 1)
    elif form == "rows_inner":
        rows = slice(n // 3, 2 * n // 3)
    dC = torch.full((rows.stop - rows.start, k), float("nan"), dtype=torch.float64, device="cuda")
    b, c = dB.data_ptr(), dC.data_ptr()
    if form == "multiply":
        st = L.spmm_multiply_device(h, b, k, c, kid, s)
    elif form == "strided":
        st = L.spmm_multiply_strided_device(h, b, k, c, k, 0, k, kid, s)
    elif form == "scatter":
        st = L.spmm_multiply_scatter_device(h, b, k, 1, (C.c_void_p * 1)(c), kid, s)
    elif form == "window":
        st = L.spmm_multiply_window_device(h, b, 0, A.n_cols, k, c, kid, s)
    elif form in ("rows", "rows_inner"):
        st = L.spmm_multiply_rows_device(h, rows.start, rows.stop, b, k, c, kid, s)
    else:
        st = L.spmm_multiply_nnz_range_device(h, z0, z1, rows.start, rows.stop - 1, b, k, c, kid, s)
    torch.cuda.synchronize()
    z = (z0, z1) if form in ("nnz", "nnz_inner") else (0, nnz)
    return st, dC.cpu().numpy(), rows, z


def last_kernel():
    _, _, _cabi = _gpu()
    return (_cabi.lib().spmm_last_kernel_name() or b"").decode()


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("case", list(CASES))
def test_each_form_runs_or_refuses_each_kernel_id(oracle, tuning_reset, case, form):
    torch, _, _cabi = _gpu()
    c = CASES[case]
    rp, ci, va, n, nc = matrix(c.mat)
    B = int_B(1, nc, c.k)
    dB = torch.from_numpy(B).cuda()
    refs = {}
    with open_handle(c) as A:
        if c.mat == "hub":
            assert A.schedule()["auto_kernel"] == "merge"
        else:
            assert A.schedule()["auto_kernel"] == "rows"
        if c.mat == "fem":
            assert A.nnz >= 200_000  # the size range in which AUTO builds the tile layout
        for kid in IDS:
            want_status, want_kernel = expected(c, form, kid)
            st, got, rows, z = call(A, form, dB, c.k, kid)
            assert st == want_status, (case, form, kid, st, (_cabi.lib().spmm_last_error() or b"").decode())
            if st != OK:
                assert np.isnan(got).all(), (case, form, kid, "a refused call wrote C")
                continue
            assert last_kernel() == NAME[want_kernel], (case, form, kid, last_kernel())
            if z not in refs:
                part = va.copy()
                part[:z[0]] = 0.0
                part[z[1]:] = 0.0
                refs[z] = oracle.spmm(rp, ci, part, B, c.k)
            want = refs[z][rows]
            diff = bits(got) != bits(want)
            assert not diff.any(), (case, form, kid, int(diff.sum()), "entries differ from the oracle")


@pytest.mark.parametrize("form", ["multiply", "strided", "scatter", "window", "rows", "nnz"])
def test_calls_without_work_check_the_kernel_id(tuning_reset, form):
    """k = 0: no launch, but the id is checked as for a call with work (BSR needs no view to be refused or accepted)."""
    torch, _, _cabi = _gpu()
    rp, ci, va, n, nc = matrix("blocked")
    # the handle's state (layout, view) and k are checked only when there is work: expect what a form gives when they fit
    fits = Case("blocked", 2, layout=True, bsr=True)
    dB = torch.zeros((nc, 1), dtype=torch.float64, device="cuda")
    with open_handle(Case("blocked", 0)) as A:
        for kid in IDS:
            want, _ = expected(fits, form, kid)
            st, _, _, _ = call(A, form, dB, 0, kid)
            assert st == want, (form, kid, st)


def test_lazy_layout_counts_whole_matrix_auto_calls(tuning_reset):
    """AUTO calls through the device, strided and scatter forms that reach the row kernel count toward the lazy tile
    layout; the call after tiled.auto_after (8) of them builds it and runs the tiled kernel. Nothing else counts."""
    torch, spmm, _cabi = _gpu()
    c = Case("fem", 16)
    rp, ci, va, n, nc = matrix("fem")
    dB = {k: torch.from_numpy(int_B(2, nc, k)).cuda() for k in (2, 8, 15, 16)}

    def run(form, k, kid, want_kernel):
        st, _, _, _ = call(A, form, dB[k], k, kid)
        assert st == OK and last_kernel() == NAME[want_kernel], (form, k, kid, st, last_kernel())
        return A.tile_info()["rows_per_tile"]

    with open_handle(c) as A:
        for _ in range(10):
            for form in ("window", "rows", "nnz"):
                assert run(form, 16, AUTO, ROWS) == 0
            for form in ("multiply", "strided", "scatter"):
                assert run(form, 16, ROWS, ROWS) == 0
                assert run(form, 16, MERGE, MERGE) == 0
            assert run("multiply", 15, AUTO, ROWS) == 0  # odd k
            assert run("scatter", 2, AUTO, ROWS) == 0    # k < 4
        _cabi.tune("stream.kmax", 8)
        _cabi.tune("stream.min_nnz", 1)
        for _ in range(10):
            assert run("strided", 8, AUTO, STREAM) == 0
        _cabi.tune("reset", 0)
        for i in range(8):
            assert run(("multiply", "strided", "scatter")[i % 3], 16, AUTO, ROWS) == 0, i
        assert run("multiply", 16, AUTO, TILED) > 0
        built16 = A.tile_info()
        assert run("multiply", 8, AUTO, TILED) > 0  # rebuilt for the 8-column k-tile
        built8 = A.tile_info()
    for k, built in ((16, built16), (8, built8)):
        with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, nc), 0) as P:
            assert P.build_tiles(-1, 0, k) == built, k


def test_bsr_auto_calls_do_not_count(tuning_reset):
    """AUTO calls that run the BSR kernel (k >= 128 on a handle with a view) leave the lazy layout's counter alone."""
    torch, spmm, _cabi = _gpu()
    from sparsematrixmultiplicationmpi_b200 import generators as gen
    rp, ci, va, n, nc = csr_of_records(*gen.fem_blocked(3, 3500, 25_000, seed=4))
    assert len(va) >= 200_000
    with spmm.DeviceCSR.from_host(spmm.SparseMatrix(va, ci, rp, n, nc), 0) as A:
        assert A.build_bsr(3) == 3
        for k, runs in ((128, BSR),) * 10 + ((16, ROWS),) * 8:
            dB = torch.from_numpy(int_B(3, nc, k)).cuda()
            st, _, _, _ = call(A, "multiply", dB, k, AUTO)
            assert st == OK and last_kernel() == NAME[runs] and A.tile_info()["rows_per_tile"] == 0, (k, last_kernel())
        dB = torch.from_numpy(int_B(3, nc, 16)).cuda()
        st, _, _, _ = call(A, "multiply", dB, 16, AUTO)
        assert st == OK and A.tile_info()["rows_per_tile"] > 0
