"""Synthetic matrices of the shapes BASELINE.json names (SuiteSparse files are unavailable offline).

Host generators return coordinate records in MatrixMarket style (0-based rows/cols/vals plus a
`symmetric` flag) so they go through the same CSR build as a loaded file; the large shapes are
generated directly in HBM (DeviceCSR.banded / DeviceCSR.rmat).

cop20k_A_shaped: cop20k_A is a symmetric FEM matrix, 121,192 x 121,192 with 2,624,331 stored
entries after symmetric expansion (report/425500_Report.tex:687), mean 21.65 per row, max 81.
The generator places the unknowns on a 49 x 49 x 51 grid in x-fastest order and couples each to
a random subset of its 26 first-ring neighbours (the 27-point FEM stencil: banded rows whose
columns cluster at offsets 0, +-1, +-nx, +-nx*ny), gives ~2 % of the unknowns a wider second-ring
coupling so the longest rows reach the real matrix's ~80 entries, leaves ~1 % of the rows empty,
and trims the edge list so the expanded count is exactly the requested nnz.
"""
from __future__ import annotations

import numpy as np


def uniform_random(n: int = 10_000, nnz_per_row: int = 10, seed: int = 1):
    """cfg1: n x n, exactly nnz_per_row distinct columns per row, values U[0.5,1.5)."""
    rng = np.random.default_rng(seed)
    rows = np.repeat(np.arange(n, dtype=np.int32), nnz_per_row)
    cols = np.empty(n * nnz_per_row, dtype=np.int32)
    # distinct columns per row: stratified draw over nnz_per_row equal strata, then a per-row rotation
    width = n // nnz_per_row
    strata = (np.arange(nnz_per_row, dtype=np.int64) * width)[None, :]
    off = rng.integers(0, width, size=(n, nnz_per_row))
    rot = rng.integers(0, n, size=(n, 1))
    cols[:] = ((strata + off + rot) % n).astype(np.int32).reshape(-1)
    vals = 0.5 + rng.random(n * nnz_per_row)
    return n, n, rows, cols, vals, False


def cop20k_A_shaped(n: int = 121_192, nnz: int = 2_624_331, seed: int = 20, nx: int = 49, ny: int = 49,
                    empty_fraction: float = 0.01, hub_fraction: float = 0.02, hub_links: int = 44,
                    max_row: int = 81):
    """Lower-triangle records of a symmetric FEM-like matrix whose expansion has exactly `nnz` entries."""
    rng = np.random.default_rng(seed)
    ids = np.arange(n, dtype=np.int64)
    x, y, z = ids % nx, (ids // nx) % ny, ids // (nx * ny)
    alive = rng.random(n) >= empty_fraction

    def ring(radius_lo, radius_hi):
        offs = []
        for dz in range(-radius_hi, radius_hi + 1):
            for dy in range(-radius_hi, radius_hi + 1):
                for dx in range(-radius_hi, radius_hi + 1):
                    r = max(abs(dx), abs(dy), abs(dz))
                    if radius_lo <= r <= radius_hi and (dz, dy, dx) < (0, 0, 0):
                        offs.append((dx, dy, dz))
        return offs

    def candidates(nodes, offs):
        src, dst = [], []
        for dx, dy, dz in offs:
            xx, yy, zz = x[nodes] + dx, y[nodes] + dy, z[nodes] + dz
            j = xx + nx * (yy + ny * zz)
            ok = (xx >= 0) & (xx < nx) & (yy >= 0) & (yy < ny) & (zz >= 0) & (j >= 0) & (j < n)
            ok &= alive[nodes] & alive[np.clip(j, 0, n - 1)]
            src.append(nodes[ok])
            dst.append(j[ok])
        return np.concatenate(src), np.concatenate(dst)

    # second-ring links of the hub unknowns (lower and upper partners, stored as (max, min))
    hubs = ids[alive & (rng.random(n) < hub_fraction)]
    hs, hd = candidates(hubs, ring(2, 2))
    hs2, hd2 = candidates(hubs, [(-dx, -dy, -dz) for dx, dy, dz in ring(2, 2)])
    hs, hd = np.concatenate([hs, hs2]), np.concatenate([hd, hd2])
    keep = rng.random(hs.size) < hub_links / 98.0
    hub_edges = np.unique(np.stack([np.maximum(hs, hd)[keep], np.minimum(hs, hd)[keep]], axis=1), axis=0)

    diag = ids[alive]
    fs, fd = candidates(ids, ring(1, 1))
    need = (nnz - diag.size - 2 * hub_edges.shape[0]) // 2
    if (nnz - diag.size) % 2:  # parity: drop one diagonal entry so 2*edges + diagonals == nnz
        diag = diag[1:]
        need = (nnz - diag.size - 2 * hub_edges.shape[0]) // 2
    if not 0 < need <= fs.size:
        raise ValueError("requested nnz does not fit the first-ring stencil")
    pick = rng.permutation(fs.size)[:need]
    er = np.concatenate([fs[pick], hub_edges[:, 0], diag])
    ec = np.concatenate([fd[pick], hub_edges[:, 1], diag])

    # cap the longest rows (degree counts both endpoints) by moving surplus edges back to unused first-ring slots
    deg = np.bincount(er, minlength=n) + np.bincount(ec, minlength=n) - np.bincount(diag, minlength=n)
    if deg.max() > max_row:
        over = np.flatnonzero(deg > max_row)
        drop = np.zeros(er.size, dtype=bool)
        for i in over:
            mine = np.flatnonzero(((er == i) | (ec == i)) & (er != ec) & ~drop)
            drop[rng.permutation(mine)[:deg[i] - max_row]] = True
        spare = np.setdiff1d(np.arange(fs.size), pick, assume_unique=False)
        add = rng.permutation(spare)[:int(drop.sum())]
        er = np.concatenate([er[~drop], fs[add]])
        ec = np.concatenate([ec[~drop], fd[add]])
    vals = 0.5 + rng.random(er.size)
    order = rng.permutation(er.size)  # file order is arbitrary; the CSR build must sort it
    return n, n, er[order].astype(np.int32), ec[order].astype(np.int32), vals[order], True


def fem_blocked(dof: int, n_nodes: int, node_nnz: int, seed: int = 20):
    """A FEM matrix with `dof` unknowns per mesh node: the node graph of cop20k_A_shaped(n_nodes, node_nnz, seed), every
    node coupling expanded into a dense dof x dof block with values U[0.5, 1.5). Returns *general* records (the lower
    triangle of the node graph mirrored here; symmetric records would be mirrored again inside the diagonal blocks).
    Node sizes of cfg2's size: dof 3: 40,397 nodes, 291,592 entries; dof 4: 30,298, 164,020; dof 6: 20,199, 72,898."""
    n, _, r, c, _, _ = cop20k_A_shaped(n=n_nodes, nnz=node_nnz, seed=seed)
    off = r != c
    nr = np.concatenate([r, c[off]]).astype(np.int64)
    nc = np.concatenate([c, r[off]]).astype(np.int64)
    i, j = np.meshgrid(np.arange(dof), np.arange(dof), indexing="ij")
    rows = (nr[:, None] * dof + i.reshape(1, -1)).reshape(-1)
    cols = (nc[:, None] * dof + j.reshape(1, -1)).reshape(-1)
    vals = 0.5 + np.random.default_rng(seed + 1).random(rows.size)
    return n * dof, n * dof, rows.astype(np.int32), cols.astype(np.int32), vals, False


def expanded_nnz(rows, cols, symmetric: bool) -> int:
    return int(rows.size + (np.count_nonzero(rows != cols) if symmetric else 0))


def write_matrix_market(path: str, n_rows, n_cols, rows, cols, vals, symmetric=False, pattern=False) -> None:
    """Coordinate file the reference loader (utils.cpp:70-185) ingests; %.17g round-trips every double."""
    kind = "pattern" if pattern else "real"
    with open(path, "w") as f:
        f.write(f"%%MatrixMarket matrix coordinate {kind} {'symmetric' if symmetric else 'general'}\n")
        f.write(f"{n_rows} {n_cols} {len(rows)}\n")
        if pattern:
            for r, c in zip(rows, cols):
                f.write(f"{r + 1} {c + 1}\n")
        else:
            for r, c, v in zip(rows, cols, vals):
                f.write(f"{r + 1} {c + 1} {v:.17g}\n")
