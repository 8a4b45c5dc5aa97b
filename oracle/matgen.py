"""oracle/matgen.py -- TEST INFRASTRUCTURE (CPU, numpy).

Synthetic matrix generators used to feed IDENTICAL CRS arrays to the oracle
and to the CUDA path (SURVEY.md F9: within-row order decides summation order).
The product has its own device-side generators
(basic_iterative_solvers_b200/csrc/bis_generate.cu); tests compare them with
these.

HPCG-n (SURVEY.md 8(d)): 27-point stencil on an nx*ny*nz grid, natural order
row = (z*ny + y)*nx + x, A_ii = 26, A_ij = -1 for the in-grid neighbours,
columns ascending inside a row.

Anderson (stand-in for SCAMAC's generator, which is absent: `parity
unpinned` for the matrix CONTENT, see DESIGN.md): 3-D 7-point, hopping -t,
on-site diagonal ranpot * U(-1, 1) from splitmix64(seed, row), open or
periodic boundaries, columns ascending inside a row.
"""
from __future__ import annotations

import numpy as np

_GOLDEN = np.uint64(0x9E3779B97F4A7C15)
_M1 = np.uint64(0xBF58476D1CE4E5B9)
_M2 = np.uint64(0x94D049BB133111EB)


def splitmix64_unit(seed: int, idx: np.ndarray) -> np.ndarray:
    """u in [0,1): splitmix64 finaliser of seed + (idx+1)*golden, top 53 bits."""
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + (idx.astype(np.uint64) + np.uint64(1)) * _GOLDEN
        z = (z ^ (z >> np.uint64(30))) * _M1
        z = (z ^ (z >> np.uint64(27))) * _M2
        z = z ^ (z >> np.uint64(31))
    return (z >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def hpcg(nx: int, ny: int | None = None, nz: int | None = None,
         row_begin: int = 0, row_end: int | None = None, index_dtype=np.int32):
    """CRS (row_ptr, col, val) of rows [row_begin,row_end) with GLOBAL columns."""
    ny = nx if ny is None else ny
    nz = nx if nz is None else nz
    n = nx * ny * nz
    row_end = n if row_end is None else row_end
    rows = np.arange(row_begin, row_end, dtype=np.int64)
    x = rows % nx
    y = (rows // nx) % ny
    z = rows // (nx * ny)
    m = rows.size
    cols = np.empty((m, 27), dtype=np.int64)
    valid = np.empty((m, 27), dtype=bool)
    vals = np.empty((m, 27), dtype=np.float64)
    k = 0
    for dz in (-1, 0, 1):
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                ok = ((x + dx >= 0) & (x + dx < nx) & (y + dy >= 0) & (y + dy < ny)
                      & (z + dz >= 0) & (z + dz < nz))
                cols[:, k] = rows + (dz * ny + dy) * nx + dx
                valid[:, k] = ok
                vals[:, k] = 26.0 if (dx == 0 and dy == 0 and dz == 0) else -1.0
                k += 1
    counts = valid.sum(axis=1)
    row_ptr = np.zeros(m + 1, dtype=np.int64)
    np.cumsum(counts, out=row_ptr[1:])
    col = cols[valid].astype(np.int32)
    val = vals[valid]
    return row_ptr.astype(index_dtype), col, val


def hpcg_nnz(nx, ny=None, nz=None):
    ny = nx if ny is None else ny
    nz = nx if nz is None else nz
    return (3 * nx - 2) * (3 * ny - 2) * (3 * nz - 2)


def anderson_diagonal(rows: np.ndarray, ranpot: float = 5.0, seed: int = 1) -> np.ndarray:
    """on-site potential of the given rows: ranpot * U(-1, 1)"""
    return ranpot * (2.0 * splitmix64_unit(seed, rows) - 1.0)


def anderson(lx: int, ly: int, lz: int, ranpot: float = 5.0, t: float = 1.0,
             seed: int = 1, periodic: bool = False, row_begin: int = 0,
             row_end: int | None = None):
    n = lx * ly * lz
    row_end = n if row_end is None else row_end
    rows = np.arange(row_begin, row_end, dtype=np.int64)
    x = rows % lx
    y = (rows // lx) % ly
    z = rows // (lx * ly)
    m = rows.size
    cols = np.empty((m, 7), dtype=np.int64)
    valid = np.empty((m, 7), dtype=bool)
    vals = np.empty((m, 7), dtype=np.float64)
    diag = anderson_diagonal(rows, ranpot, seed)
    steps = [(0, 0, -1), (0, -1, 0), (-1, 0, 0), (0, 0, 0), (1, 0, 0), (0, 1, 0), (0, 0, 1)]
    for k, (dx, dy, dz) in enumerate(steps):
        xx, yy, zz = x + dx, y + dy, z + dz
        if periodic:
            ok = np.ones(m, dtype=bool)
            # a dimension of length 1 or 2 would duplicate entries: drop wrap there
            if lx <= 2 and dx:
                ok &= (xx >= 0) & (xx < lx)
            if ly <= 2 and dy:
                ok &= (yy >= 0) & (yy < ly)
            if lz <= 2 and dz:
                ok &= (zz >= 0) & (zz < lz)
            xx, yy, zz = xx % lx, yy % ly, zz % lz
        else:
            ok = (xx >= 0) & (xx < lx) & (yy >= 0) & (yy < ly) & (zz >= 0) & (zz < lz)
        cols[:, k] = (zz * ly + yy) * lx + xx
        valid[:, k] = ok
        vals[:, k] = diag if (dx, dy, dz) == (0, 0, 0) else -t
    if periodic:
        big = np.iinfo(np.int64).max
        key = np.where(valid, cols, big)
        order = np.argsort(key, axis=1, kind="stable")
        cols = np.take_along_axis(cols, order, axis=1)
        vals = np.take_along_axis(vals, order, axis=1)
        valid = np.take_along_axis(valid, order, axis=1)
    counts = valid.sum(axis=1)
    row_ptr = np.zeros(m + 1, dtype=np.int64)
    np.cumsum(counts, out=row_ptr[1:])
    return row_ptr.astype(np.int32), cols[valid].astype(np.int32), vals[valid]


def random_spd(n: int, nnz_per_row: int = 5, seed: int = 0, shuffle_cols: bool = True):
    """Ragged, unsorted-column, strictly diagonally dominant symmetric matrix."""
    rng = np.random.default_rng(seed)
    import scipy.sparse as sp
    rows = np.repeat(np.arange(n), nnz_per_row)
    cols = rng.integers(0, n, size=rows.size)
    v = rng.uniform(-1.0, 1.0, size=rows.size)
    a = sp.coo_matrix((v, (rows, cols)), shape=(n, n)).tocsr()
    a = a + a.T
    a.setdiag(0.0)
    a.eliminate_zeros()
    d = np.abs(a).sum(axis=1).A1 + 1.0 + rng.uniform(0, 1, n)
    a = (a + sp.diags(d)).tocsr()
    a.sort_indices()
    rp, col, val = a.indptr.astype(np.int32), a.indices.astype(np.int32), a.data.copy()
    if shuffle_cols:
        for r in range(n):
            s, e = rp[r], rp[r + 1]
            p = rng.permutation(e - s)
            col[s:e] = col[s:e][p]
            val[s:e] = val[s:e][p]
    return rp, col, val


def random_general(n: int, nnz_per_row: int = 6, seed: int = 0):
    """Nonsymmetric, diagonally dominant, ragged rows (some rows diag only)."""
    rng = np.random.default_rng(seed)
    import scipy.sparse as sp
    lens = rng.integers(0, 2 * nnz_per_row, size=n)
    rows = np.repeat(np.arange(n), lens)
    cols = rng.integers(0, n, size=rows.size)
    v = rng.uniform(-1.0, 1.0, size=rows.size)
    a = sp.coo_matrix((v, (rows, cols)), shape=(n, n)).tocsr()
    a.setdiag(0.0)
    a.eliminate_zeros()
    d = np.abs(a).sum(axis=1).A1 + 1.0 + rng.uniform(0, 1, n)
    a = (a + sp.diags(d)).tocsr()
    a.sort_indices()
    return a.indptr.astype(np.int32), a.indices.astype(np.int32), a.data.copy()
