"""The oracle (oracle/spmm_oracle.c) against the reference's golden vectors and the compiled reference itself."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, random_csr

CASES = ["small", "hub", "k1", "k8"]


def test_kat_report_example(oracle, golden_multiply):
    g = golden_multiply
    # SURVEY.md Appendix A.1 (report/425500_Report.tex:208-223 with generateLargeFatVector(4,3))
    assert g["kat_B"].tolist() == [[84, 87, 78], [16, 94, 36], [87, 93, 50], [22, 63, 28]]
    assert g["kat_C"].tolist() == [[258, 273, 178], [261, 279, 150], [0, 0, 0], [88, 252, 112]]
    for strat, P in [("seq", 1), ("row", 2), ("col", 2), ("nnz", 3)]:
        C = oracle.spmm(g["kat_rowptr"], g["kat_colidx"], g["kat_vals"], g["kat_B"], 3, strat, P)
        assert np.array_equal(C, g["kat_C"])


def test_fat_vector_generator(oracle, golden_multiply):
    assert np.array_equal(oracle.generate_fatvector(7, 5), golden_multiply["fatvec_7x5"])
    assert np.array_equal(oracle.generate_fatvector(4, 3), golden_multiply["kat_B"])


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_golden_bitwise(oracle, golden_multiply, name):
    g = golden_multiply
    a = (g[f"{name}_rowptr"], g[f"{name}_colidx"], g[f"{name}_vals"], g[f"{name}_B"])
    k = a[3].shape[1]
    assert np.array_equal(oracle.spmm(*a, k, "seq"), g[f"{name}_C_seq"])
    for P in (2, 3, 7):
        for strat in ("row", "col", "nnz"):
            assert np.array_equal(oracle.spmm(*a, k, strat, P), g[f"{name}_C_{strat}_P{P}"]), (strat, P)
        # SURVEY.md F7: row-wise and column-wise are bit-identical to sequential for every P
        assert np.array_equal(g[f"{name}_C_row_P{P}"], g[f"{name}_C_seq"])
        assert np.array_equal(g[f"{name}_C_col_P{P}"], g[f"{name}_C_seq"])
        assert np.allclose(g[f"{name}_C_nnz_P{P}"], g[f"{name}_C_seq"], rtol=0, atol=1e-9)


@pytest.mark.parametrize("seed,n,mean,k,P", [(1, 300, 6, 4, 4), (2, 257, 15, 1, 5), (3, 64, 3, 7, 9), (4, 5, 2, 3, 6)])
def test_oracle_matches_compiled_reference(oracle, reference, seed, n, mean, k, P):
    rowptr, colidx, vals = random_csr(seed, n, n, mean, long_row=min(4 * n, 900), empty_every=5)
    B = np.random.default_rng(seed).integers(1, 101, (n, k)).astype(np.float64)
    for strat in ("seq", "row", "col", "nnz"):
        ref, _ = reference.spmm(n, rowptr, colidx, vals, B, k, strat, P)
        assert np.array_equal(oracle.spmm(rowptr, colidx, vals, B, k, strat, P), ref), strat


def test_partitions_match_reference_formulas(oracle):
    for total, P in [(10, 3), (5, 6), (121192, 8), (0, 4), (7, 7), (2624331, 5)]:
        rows = [oracle.partition("rows", total, P, r) for r in range(P)]
        assert rows[0][0] == 0 and rows[-1][1] == total and all(rows[i][1] == rows[i + 1][0] for i in range(P - 1))
        assert max(e - s for s, e in rows) - min(e - s for s, e in rows) <= 1
        cols = [oracle.partition("cols", total, P, r) for r in range(P)]
        assert cols[-1][1] == total and all(e - s == total // P for s, e in cols[:-1])  # last rank takes the extras
        nz = [oracle.partition("nnz", total, P, r) for r in range(P)]
        assert nz[0][0] == 0 and nz[-1][1] == total and all(nz[i][1] == nz[i + 1][0] for i in range(P - 1))


LOADER = ["general_unsorted", "symmetric", "pattern", "duplicates", "skew_symmetric", "rectangular",
          "pattern_symmetric", "empty_rows", "random_symmetric"]


@pytest.mark.parametrize("name", LOADER)
def test_oracle_loader_matches_reference_golden(oracle, golden_loader, name):
    nr, nc, rp, ci, va = oracle.read_mtx(os.path.join(GOLDEN, name + ".mtx"))
    g = golden_loader
    assert [nr, nc] == g[f"{name}_shape"].tolist()
    assert np.array_equal(rp, g[f"{name}_rowptr"])
    assert np.array_equal(ci, g[f"{name}_colidx"])
    assert np.array_equal(va.view(np.uint64), g[f"{name}_vals"].view(np.uint64))  # bit-exact


def test_loader_appendix_a2_values(golden_loader):
    g = golden_loader
    assert g["general_unsorted_rowptr"].tolist() == [0, 2, 3, 4] and g["general_unsorted_colidx"].tolist() == [0, 2, 1, 0]
    assert g["general_unsorted_vals"].tolist() == [1, 2, -0.3, 5.5]
    assert g["symmetric_colidx"].tolist() == [0, 1, 2, 0, 0, 2] and g["symmetric_vals"].tolist() == [1, 2, 3, 2, 3, 4]
    assert g["duplicates_colidx"].tolist() == [0, 1, 1, 1] and g["duplicates_vals"].tolist() == [7, 1, 9, 1]
    assert g["skew_symmetric_vals"].tolist() == [5, 5]  # treated as symmetric, no sign flip
    assert g["rectangular_shape"].tolist() == [2, 4]


def test_loader_errors(oracle, tmp_path):
    with pytest.raises(RuntimeError, match="Unable to open file"):
        oracle.read_mtx(str(tmp_path / "missing.mtx"))
    p = tmp_path / "short.mtx"
    p.write_text("%%MatrixMarket matrix coordinate real general\n3 3 4\n1 1 1\n2 2 2\n")
    with pytest.raises(RuntimeError, match="Failed to read data"):
        oracle.read_mtx(str(p))


def test_loader_against_compiled_reference_on_generated_file(oracle, reference, tmp_path):
    from sparsematrixmultiplicationmpi_b200 import generators as gen
    n, _, r, c, v, sym = gen.cop20k_A_shaped(n=3000, nnz=60001, nx=12, ny=12, seed=3)
    path = str(tmp_path / "fem.mtx")
    gen.write_matrix_market(path, n, n, r, c, v, symmetric=sym)
    a = oracle.read_mtx(path)
    b = reference.read_mtx(path)
    assert a[0] == b[0] and a[1] == b[1]
    for x, y in zip(a[2:], b[2:]):
        assert np.array_equal(x, y)
    assert a[2][-1] == 60001


def test_are_equal_and_serialize(oracle):
    """areMatricesEqual's verdicts on either side of its bound; the compiled reference, where oracle/_ref is built, gives the same."""
    import pyoracle
    checkers = [oracle] + ([pyoracle.Reference("exact")] if pyoracle.Reference.available() else [])
    a = np.arange(12, dtype=np.float64).reshape(4, 3)
    b = a.copy()
    b[2, 1] += 5e-7
    assert all(x.are_equal(a, b, 1e-6) for x in checkers)
    b[2, 1] += 1e-6
    assert not any(x.are_equal(a, b, 1e-6) for x in checkers)
    if len(checkers) > 1:
        assert checkers[1].serialize_is_rowmajor(a, 4, 3)
