"""Host-side logic that needs no GPU: partitions, utils mirrors, MatrixMarket front end, generators, shards."""
import math
import os

import numpy as np
import pytest

import sparsematrixmultiplicationmpi_b200 as spmm
from sparsematrixmultiplicationmpi_b200 import _cabi, generators as gen
from sparsematrixmultiplicationmpi_b200.strategies import NonZeroRanges
from conftest import GOLDEN, random_csr


@pytest.mark.parametrize("total,P", [(10, 3), (5, 6), (121192, 8), (0, 4), (7, 7), (2624331, 5), (64, 64)])
def test_partitions_equal_oracle(oracle, total, P):
    for r in range(P):
        assert spmm.partition_rows(total, P, r) == oracle.partition("rows", total, P, r) == _cabi.partition_rows(total, P, r)
        assert spmm.partition_cols(total, P, r) == oracle.partition("cols", total, P, r) == _cabi.partition_cols(total, P, r)
        assert spmm.partition_nnz(total, P, r) == oracle.partition("nnz", total, P, r) == _cabi.partition_nnz(total, P, r)


def test_retired_tuning_keys_are_rejected():
    """Keys of kernel variants that were removed fail loudly instead of being ignored."""
    for key, value in (("rows.sweep", 1), ("tiled.kt", 32)):
        with pytest.raises(_cabi.SpmmError) as e:
            _cabi.tune(key, value)
        assert e.value.status == _cabi.SPMM_ERR_INVALID


def test_generate_fat_vector_is_the_reference_sequence(golden_multiply):
    assert np.array_equal(spmm.generateLargeFatVector(4, 3), golden_multiply["kat_B"])
    assert np.array_equal(spmm.generateLargeFatVector(7, 5), golden_multiply["fatvec_7x5"])
    assert np.array_equal(spmm.generateLargeFatVector(7, 5), spmm.generateLargeFatVector(7, 5))


def test_serialize_roundtrip_and_compare():
    a = spmm.generateLargeFatVector(6, 4)
    flat = spmm.serialize(a)
    assert flat.shape == (24,) and np.array_equal(flat, a.reshape(-1))
    assert np.array_equal(spmm.deserialize(flat, 6, 4), a)
    b = a.copy()
    b[3, 2] += 5e-7
    assert spmm.areMatricesEqual(a, b, 1e-6)
    b[3, 2] += 1e-6
    assert not spmm.areMatricesEqual(a, b, 1e-6)
    assert not spmm.areMatricesEqual(a, a[:5], 1e-6)


@pytest.mark.parametrize("name", ["general_unsorted", "symmetric", "pattern", "duplicates", "skew_symmetric",
                                  "rectangular", "pattern_symmetric", "empty_rows", "random_symmetric"])
def test_matrix_market_front_end_feeds_the_same_records(oracle, golden_loader, name):
    path = os.path.join(GOLDEN, name + ".mtx")
    nr, nc, rows, cols, vals, sym = spmm.parse_matrix_market(path)
    onr, onc, orows, ocols, ovals, osym, _ = oracle.read_mtx_coo(path)
    assert (nr, nc, sym) == (onr, onc, osym)
    assert np.array_equal(rows, orows) and np.array_equal(cols, ocols)
    assert np.array_equal(vals.view(np.uint64), ovals.view(np.uint64))
    # and the oracle's CSR assembly of those records is the reference loader's output
    rp, ci, va = oracle.csr_from_coo(nr, rows, cols, vals, sym)
    assert np.array_equal(rp, golden_loader[f"{name}_rowptr"]) and np.array_equal(ci, golden_loader[f"{name}_colidx"])


def test_matrix_market_errors(tmp_path):
    with pytest.raises(RuntimeError, match="Unable to open file"):
        spmm.parse_matrix_market(str(tmp_path / "nope.mtx"))
    p = tmp_path / "short.mtx"
    p.write_text("%%MatrixMarket matrix coordinate real general\n3 3 4\n1 1 1\n2 2 2\n")
    with pytest.raises(RuntimeError, match="Failed to read data"):
        spmm.parse_matrix_market(str(p))
    p2 = tmp_path / "nosize.mtx"
    p2.write_text("%%MatrixMarket matrix coordinate real general\n")
    with pytest.raises(RuntimeError, match="Failed to read matrix dimensions"):
        spmm.parse_matrix_market(str(p2))


def test_matrix_market_native_reader_token_stream(oracle, tmp_path):
    """The body is a token stream (utils.cpp:128-136): records may span lines, '+' signs, CRLF, tabs; a file large
    enough for several reader threads must give the oracle's records bit for bit."""
    p = tmp_path / "odd.mtx"
    p.write_bytes(b"%%MatrixMarket matrix coordinate real general\r\n% a comment\r\n3 4 4\r\n1 1\n2.5 2\t+3 -1e-3\r\n"
                  b"3 4 0x1p-1 1\n\n 2 +7.25E+1\n trailing tokens are ignored 9 9 9\n")
    nr, nc, rows, cols, vals, sym = spmm.parse_matrix_market(str(p))
    assert (nr, nc, sym) == (3, 4, False)
    assert rows.tolist() == [0, 1, 2, 0] and cols.tolist() == [0, 2, 3, 1]
    assert vals.tolist() == [2.5, -1e-3, 0.5, 72.5]
    rng = np.random.default_rng(5)
    n, ne = 4000, 300_000
    r, c = rng.integers(1, n + 1, ne), rng.integers(1, n + 1, ne)
    v = rng.standard_normal(ne) * 10.0 ** rng.integers(-30, 30, ne)
    big = tmp_path / "big.mtx"
    with open(big, "w") as f:
        f.write("%%MatrixMarket matrix coordinate real symmetric\n%c\n")
        f.write(f"{n} {n} {ne}\n")
        f.write("".join(f"{a} {b} {float(x)!r}" + ("\n" if i % 3 else " ") for i, (a, b, x) in enumerate(zip(r, c, v))))
    nr, nc, rows, cols, vals, sym = spmm.parse_matrix_market(str(big))
    onr, onc, orows, ocols, ovals, osym, _ = oracle.read_mtx_coo(str(big))
    assert (nr, nc, sym) == (onr, onc, osym) == (n, n, True)
    assert np.array_equal(rows, orows) and np.array_equal(cols, ocols)
    assert np.array_equal(vals.view(np.uint64), ovals.view(np.uint64))
    assert np.array_equal(vals, v)  # repr() round-trips every double
    for junk in ("2 x 3.0", "2 2 +-3.0", "+-2 2 3.0", "2 2 3.0.1", "2 2 1e"):
        bad = tmp_path / "bad.mtx"
        bad.write_text("%%MatrixMarket matrix coordinate real general\n2 2 2\n1 1 1.0\n" + junk + "\n")
        with pytest.raises(RuntimeError, match="Failed to read data"):
            spmm.parse_matrix_market(str(bad))
        with pytest.raises(RuntimeError, match="Failed to read data"):
            oracle.read_mtx_coo(str(bad))
    oob = tmp_path / "oob.mtx"
    oob.write_text("%%MatrixMarket matrix coordinate real general\n2 2 1\n3 1 1.0\n")
    with pytest.raises(RuntimeError, match="outside the declared"):
        spmm.parse_matrix_market(str(oob))


def test_matrix_market_native_reader_random_token_layouts(oracle, tmp_path):
    """Property test: whatever the whitespace between tokens and the spelling of the numbers, the native reader and the
    oracle's restatement of utils.cpp:70-153 produce the same records, bit for bit."""
    hypothesis = pytest.importorskip("hypothesis")
    from hypothesis import given, settings, strategies as st

    seps = st.sampled_from([" ", "  ", "\t", "\n", " \n", "\r\n", "\n\n", " \t "])
    spell = st.sampled_from(["{!r}", "{:.17g}", "{:.17e}", "+{:.17g}", "{:.20f}"])

    @settings(max_examples=60, deadline=None)
    @given(st.integers(1, 40), st.integers(1, 40), st.integers(0, 60), st.booleans(), st.booleans(), st.data())
    def check(nr, nc, ne, symmetric, pattern, data):
        if symmetric:
            nc = nr
        rows = data.draw(st.lists(st.integers(1, nr), min_size=ne, max_size=ne))
        cols = data.draw(st.lists(st.integers(1, nc), min_size=ne, max_size=ne))
        vals = data.draw(st.lists(st.floats(-1e30, 1e30, allow_nan=False, width=64), min_size=ne, max_size=ne))
        kind = "pattern" if pattern else "real"
        text = f"%%MatrixMarket matrix coordinate {kind} {'symmetric' if symmetric else 'general'}\n% comment\n{nr} {nc} {ne}\n"
        for r, c, v in zip(rows, cols, vals):
            text += f"{r}{data.draw(seps)}{c}"
            if not pattern:
                fmt = data.draw(spell)
                # "+" only in front of a number whose own spelling carries no sign (-0.0 >= 0 is true, and "+-0" is a
                # token reference, oracle and native reader all reject)
                positive = math.copysign(1.0, v) > 0
                text += data.draw(seps) + (fmt if positive or not fmt.startswith("+") else "{!r}").format(float(v))
            text += data.draw(seps)
        path = tmp_path / "prop.mtx"
        path.write_text(text, newline="")
        both_fail_or_agree(path)

    def both_fail_or_agree(path):
        """Product and oracle accept the same files: either both raise, or their records are bit-equal."""
        try:
            expected = oracle.read_mtx_coo(str(path))
        except RuntimeError:
            with pytest.raises(RuntimeError):
                spmm.parse_matrix_market(str(path))
            return
        got = spmm.parse_matrix_market(str(path))
        onr, onc, orows, ocols, ovals, osym, _ = expected
        assert (got[0], got[1], got[5]) == (onr, onc, osym)
        assert np.array_equal(got[2], orows) and np.array_equal(got[3], ocols)
        assert np.array_equal(got[4].view(np.uint64), ovals.view(np.uint64))

    check()
    # malformed value tokens: both sides must refuse them together
    for bad in ("+-0", "+-1.5", "1.5x", "--2"):
        path = tmp_path / "bad.mtx"
        path.write_text(f"%%MatrixMarket matrix coordinate real general\n2 2 1\n1 1 {bad}\n")
        both_fail_or_agree(path)


def test_cop20k_shaped_generator_hits_the_published_shape():
    n, nc, r, c, v, sym = gen.cop20k_A_shaped()
    assert (n, nc, sym) == (121192, 121192, True)
    assert gen.expanded_nnz(r, c, sym) == 2624331  # report/425500_Report.tex:687
    assert np.all(r >= c)  # lower triangle, MatrixMarket symmetric storage
    deg = np.bincount(r, minlength=n) + np.bincount(c, minlength=n) - np.bincount(r[r == c], minlength=n)
    assert deg.max() <= 81 and (deg == 0).sum() > 0
    assert np.all((v >= 0.5) & (v < 1.5))
    # banded: columns sit within +-2 grid planes (+ ring) of the diagonal
    assert np.max(r - c) <= 2 * 49 * 49 + 2 * 49 + 2


def test_uniform_random_generator_cfg1():
    n, _, r, c, v, sym = gen.uniform_random(10_000, 10, seed=1)
    assert r.size == 100_000 and not sym
    key = r.astype(np.int64) * n + c
    assert np.unique(key).size == key.size  # distinct columns in every row


def test_nnz_shards_tile_the_stream(oracle):
    rowptr, colidx, vals = random_csr(5, 120, 120, 6, long_row=700, empty_every=4)
    m = spmm.SparseMatrix(vals, colidx, rowptr, 120, 120)
    B = np.random.default_rng(1).integers(1, 101, (120, 3)).astype(np.float64)
    for P in (1, 2, 5, 16):
        total = np.zeros((120, 3))
        covered = 0
        for r in range(P):
            local, first, last, mid = NonZeroRanges.shard_of(m, P, r)
            b, e = spmm.partition_nnz(m.nnz, P, r)
            covered += local.nnz
            assert local.nnz == e - b
            if local.nnz:
                assert mid == (b > rowptr[first])
                part = oracle.spmm(local.rowPtr, local.colIndices, local.values, B, 3)
                total[first:last + 1] += part
        assert covered == m.nnz
        assert np.allclose(total, oracle.spmm(rowptr, colidx, vals, B, 3), rtol=1e-13, atol=1e-9)


def test_product_package_never_touches_the_oracle():
    """No file of the package may import, load or name anything under oracle/ (parity would be void)."""
    pkg = os.path.dirname(spmm.__file__)
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "pyoracle" not in text and "liboracle" not in text and "oracle_spmm" not in text, f
