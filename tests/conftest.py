import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
GOLDEN = os.path.join(ROOT, "tests", "golden")

REL_TOL = 1e-12  # BASELINE.json north_star: FP64 relative tolerance per entry vs the reference's sequential result


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    import pyoracle
    return pyoracle.Oracle()


@pytest.fixture(scope="session")
def reference():
    """The reference's own code compiled into oracle/_ref by oracle/Makefile; only where its sources were given (REF=<dir>)."""
    import pyoracle
    if not pyoracle.Reference.available():
        pytest.skip("oracle/_ref not built (needs /root/reference at build time)")
    return pyoracle.Reference("exact")


@pytest.fixture(scope="session")
def golden_multiply():
    return np.load(os.path.join(GOLDEN, "multiply.npz"))


@pytest.fixture(scope="session")
def golden_loader():
    return np.load(os.path.join(GOLDEN, "loader.npz"))


def random_csr(seed, n_rows, n_cols, mean_len, long_row=None, empty_every=0, positive=False):
    """Seeded CSR with ascending (possibly duplicated) columns, optional hub row and empty rows."""
    rng = np.random.default_rng(seed)
    lens = rng.poisson(mean_len, n_rows)
    if empty_every:
        lens[::empty_every] = 0
    if long_row is not None and n_rows:
        lens[n_rows // 2] = long_row
    rowptr = np.concatenate(([0], np.cumsum(lens))).astype(np.int32)
    nnz = int(rowptr[-1])
    colidx = np.sort(rng.integers(0, max(n_cols, 1), nnz).astype(np.int32))
    # sort inside each row only
    colidx = rng.integers(0, max(n_cols, 1), nnz).astype(np.int32)
    for i in range(n_rows):
        colidx[rowptr[i]:rowptr[i + 1]].sort()
    vals = (0.5 + rng.random(nnz)) if positive else rng.standard_normal(nnz)
    return rowptr, colidx, vals


def assert_close_rel(got, ref, rowptr=None, colidx=None, vals=None, B=None, tol=REL_TOL):
    """Per-entry |x-ref| <= tol*|ref|; with mixed-sign data the bound is taken against sum_j |a_ij*b_jk|
    (SURVEY.md hard part 8: a cancelling entry has no meaningful relative error against itself)."""
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape
    scale = np.abs(ref)
    if rowptr is not None:
        n = len(rowptr) - 1
        absC = np.zeros_like(ref)
        rows = np.repeat(np.arange(n), np.diff(rowptr))
        np.add.at(absC, rows, np.abs(vals)[:, None] * np.abs(np.asarray(B)[colidx]))
        scale = absC
    err = np.abs(got - ref)
    bad = err > tol * scale
    assert not bad.any(), f"max err/scale = {np.max(err[bad] / np.maximum(scale[bad], 1e-300)):.3e} at {np.argwhere(bad)[0]}"
