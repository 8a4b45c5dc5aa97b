"""The slab-wise oracle (oracle/port.py: GeneratedSlabs, TemplatedSlabs, spmv_slabwise, sptrsv_slabwise) is the
reference of the GPU tests past 2^31 nonzeros, where the whole-matrix oracle cannot run (int row_ptr).  On
matrices small enough for both, the slab-wise SpMV and forward / backward triangular solves must have the bits
of the whole-matrix oracle (port.spmv, port.sptrsv on the split of o_split_strict), for every slab height --
one row, heights that do not divide the row or plane count, one slab for everything -- and the templated HPCG
and Anderson slabs must have the bits of the generated ones."""
import numpy as np
import pytest

from oracle import matgen, port

HPCG_DIMS = [(7, 5, 3), (20, 14, 11), (130, 7, 5)]
ANDERSON = {
    "open": dict(lx=9, ly=7, lz=13, ranpot=5.0, t=1.0, seed=7, periodic=False),
    "periodic": dict(lx=9, ly=7, lz=13, ranpot=5.0, t=1.0, seed=7, periodic=True),
}


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def whole_reference(rp, col, val, x, b):
    """(A x, L solve, U solve) of the whole-matrix oracle, D = diag(A) as o_split_strict extracts it"""
    f = port.factor(rp, col, val)
    y = port.spmv(rp, col, val, x)
    xl = port.sptrsv(f.l_rp, f.l_col, f.l_val, f.A_D, b)
    xu = port.sptrsv(f.u_rp, f.u_col, f.u_val, f.A_D, b, backward=True)
    return y, xl, xu, f.A_D


def check_slabs(slabs, ref, x, b):
    y, xl, xu, D = ref
    assert np.array_equal(bits(port.spmv_slabwise(slabs, x, threads=3)), bits(y))
    assert np.array_equal(bits(port.sptrsv_slabwise(slabs, D, b)), bits(xl))
    assert np.array_equal(bits(port.sptrsv_slabwise(slabs, D, b, backward=True)), bits(xu))
    diag = np.concatenate([slabs.split(rb, re)[2] for rb, re in slabs.bounds])
    assert np.array_equal(bits(diag), bits(D))


def vectors(n, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(-1.0, 1.0, n), rng.uniform(-1.0, 1.0, n)


@pytest.mark.parametrize("dims", HPCG_DIMS)
def test_hpcg_generated_slabs_match_whole_oracle(dims):
    nx, ny, nz = dims
    rp, col, val = matgen.hpcg(nx, ny, nz)
    n = rp.size - 1
    x, b = vectors(n, 1)
    ref = whole_reference(rp, col, val, x, b)
    for slab_rows in (1, 7, nx * ny + 3, 2 * nx * ny - 1, n - 1, n):
        slabs = port.GeneratedSlabs(lambda r0, r1: matgen.hpcg(nx, ny, nz, r0, r1), n, slab_rows)
        check_slabs(slabs, ref, x, b)


@pytest.mark.parametrize("dims", HPCG_DIMS)
def test_hpcg_templated_slabs_match_generated_and_whole_oracle(dims):
    nx, ny, nz = dims
    rp, col, val = matgen.hpcg(nx, ny, nz)
    n = rp.size - 1
    plane = nx * ny
    x, b = vectors(n, 2)
    ref = whole_reference(rp, col, val, x, b)
    for planes in sorted({1, 2, 4, nz - 1, nz} - {0}):
        tmpl = port.hpcg_slabs(nx, ny, nz, planes)
        gen = port.GeneratedSlabs(lambda r0, r1: matgen.hpcg(nx, ny, nz, r0, r1), n, planes * plane)
        assert tmpl.bounds == gen.bounds
        # at most three distinct slabs are generated, however many the matrix has
        assert len(tmpl._crs) <= 3 and len(tmpl._crs) <= len(tmpl.bounds)
        for rb, re in tmpl.bounds:
            for a, g in zip(tmpl.crs(rb, re), gen.crs(rb, re)):
                assert np.array_equal(a, g)
        check_slabs(tmpl, ref, x, b)


@pytest.mark.parametrize("kind", sorted(ANDERSON))
def test_anderson_generated_and_templated_slabs_match_whole_oracle(kind):
    p = ANDERSON[kind]
    rp, col, val = matgen.anderson(**p)
    n = rp.size - 1
    x, b = vectors(n, 3)
    if p["periodic"]:
        # the wrap puts a row's periodic neighbours out of stencil order: storage order is by column
        assert np.all(np.diff(col[rp[0]:rp[1]]) > 0) and col[rp[1] - 1] > p["lx"] * p["ly"]
    ref = whole_reference(rp, col, val, x, b)
    plane = p["lx"] * p["ly"]
    for slab_rows in (1, 5, plane, 3 * plane + 2, n):
        slabs = port.GeneratedSlabs(lambda r0, r1: matgen.anderson(**p, row_begin=r0, row_end=r1), n, slab_rows)
        check_slabs(slabs, ref, x, b)
    for planes in (1, 3, p["lz"] - 1):
        tmpl = port.anderson_slabs(p["lx"], p["ly"], p["lz"], planes, p["ranpot"], p["t"], p["seed"], p["periodic"])
        gen = port.GeneratedSlabs(lambda r0, r1: matgen.anderson(**p, row_begin=r0, row_end=r1), n, planes * plane)
        assert tmpl.bounds == gen.bounds and len(tmpl._crs) <= 3
        for rb, re in tmpl.bounds:
            for a, g in zip(tmpl.crs(rb, re), gen.crs(rb, re)):
                assert np.array_equal(bits(a) if a.dtype == np.float64 else a, bits(g) if g.dtype == np.float64 else g)
        check_slabs(tmpl, ref, x, b)


def test_slab_rows_start_at_zero_and_columns_rebase():
    """the slab CRS the GPU tests rely on: row_ptr from 0, int32, and columns below the slab negative"""
    nx, ny, nz = 6, 5, 4
    rb, re = 2 * nx * ny, 3 * nx * ny
    rp, col, val = port.rebase(*matgen.hpcg(nx, ny, nz, rb, re), rb)
    assert rp.dtype == np.int32 and col.dtype == np.int32 and rp[0] == 0
    assert col.min() == -nx * ny and col.max() == 2 * nx * ny - 1     # corner rows: one plane down / up
    full = matgen.hpcg(nx, ny, nz)
    assert np.array_equal(col + rb, full[1][full[0][rb]:full[0][re]])
