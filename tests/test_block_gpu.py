"""GPU tests of the multi-right-hand-side path (include/bis_b200.h, "multiple right-hand sides").

 - bis_spmm: every column bit-identical to the oracle's native_spmv, and to bis_spmv where that adds in storage order;
 - the entry points fail loudly on bad arguments;
 - block CG (host.solve_block): every column bit-identical to the single-vector composition bis_spmv /
   bis_dot_to_slot / bis_cg_update / bis_cg_direction_x with the harness's stop rule, defined here as a Python loop;
   within the north-star bar of host.solve("cg") and of the oracle; invariant under column permutation, k, graphs.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import golden
from oracle import matgen, port

from basic_iterative_solvers_b200 import capi, host

pytestmark = pytest.mark.gpu

S_RR, S_RZ_NEW, S_RZ, S_PAP = 0, 1, 2, 3


def named(name):
    if name == "hpcg16":
        return matgen.hpcg(16)
    if name == "hpcg32":
        return matgen.hpcg(32)
    g = golden(name)
    return g["rp"], g["col"], g["val"]


def unstructured(n, long_row, seed):
    """Random pattern in unsorted column order, every 7th row empty, row 3 with `long_row` nonzeros."""
    rng = np.random.default_rng(seed)
    rows = []
    for i in range(n):
        m = 0 if i % 7 == 5 else int(rng.integers(1, 12))
        if i == 3:
            m = long_row
        rows.append(rng.permutation(n)[:m].astype(np.int32))
    rp = np.zeros(n + 1, np.int32)
    rp[1:] = np.cumsum([len(r) for r in rows])
    col = np.concatenate(rows).astype(np.int32)
    val = rng.uniform(-2, 2, col.size)
    return rp, col, val


MATRICES = {
    "hpcg16": lambda: named("hpcg16"),
    "fdm2d16": lambda: named("fdm2d16"),
    "band_klein": lambda: named("band_klein"),
    "random300": lambda: named("random300"),
    "anderson": lambda: named("anderson_12_10_8"),
    "unstructured_row120": lambda: unstructured(400, 120, 3),     # TMA tiles of 32 rows
    "unstructured_row1800": lambda: unstructured(2000, 1800, 4),  # too long for a tile: the direct kernel
    "hpcg16_rp64": lambda: tuple([named("hpcg16")[0].astype(np.int64)] + list(named("hpcg16")[1:])),
}


def spmm(ctx, A, X):
    n_out = A.info()["n_rows"]
    k = X.shape[1]
    dX = ctx.upload(X)
    dY = ctx.alloc(n_out * k)
    ctx.spmm(A, dX, dY, k)
    Y = ctx.download(dY, n_out * k).reshape(n_out, k)
    ctx.free(dX), ctx.free(dY)
    return Y


@pytest.mark.parametrize("k", [1, 2, 3, 5, 8, 16])
@pytest.mark.parametrize("mat", list(MATRICES))
def test_spmm_vs_oracle_bitwise(ctx, mat, k):
    rp, col, val = MATRICES[mat]()
    n = len(rp) - 1
    A = ctx.upload_crs(rp, col, val)
    assert A.info()["rp_bytes"] == (8 if np.asarray(rp).dtype == np.int64 else 4)
    X = np.random.default_rng(k).uniform(-1, 1, (n, k))
    Y = spmm(ctx, A, X)
    for j in range(k):
        assert np.array_equal(Y[:, j], port.spmv(rp, col, val, X[:, j].copy())), (mat, k, j)
    A.free()


@pytest.mark.parametrize("vdict", [0, 1])
def test_spmm_vs_spmv_hpcg64_bitwise(ctx, vdict):
    ctx.set_option("spmv_vdict", vdict)
    try:
        A = ctx.generate_hpcg(64)
        n = A.info()["n_rows"]
        X = np.random.default_rng(11).uniform(-1, 1, (n, 8))
        Y = spmm(ctx, A, X)
        dx, dy = ctx.alloc(n), ctx.alloc(n)
        for j in range(8):
            ctx.upload(X[:, j].copy(), dx)
            ctx.call("bis_spmv", A.h, dx, dy)
            assert np.array_equal(Y[:, j], ctx.download(dy, n)), j
        if vdict:
            assert ctx.get_option("spmv_value_bytes") == 1
        ctx.free(dx), ctx.free(dy), A.free()
    finally:
        ctx.set_option("spmv_vdict", 0)


def test_block_entry_points_fail_loudly(ctx):
    rp, col, val = named("hpcg16")
    n = len(rp) - 1
    A = ctx.upload_crs(rp, col, val)
    X, Y = ctx.alloc(n * 17 + 2), ctx.alloc(n * 17)
    for k in (0, 17):
        with pytest.raises(capi.BisError):
            ctx.spmm(A, X, Y, k)
        with pytest.raises(capi.BisError):
            ctx.call("bis_block_dot_to_slots", n, k, X, Y, 40, None)
    with pytest.raises(capi.BisError):
        ctx.spmm(A, X + 8, Y, 4)                     # misaligned X
    with pytest.raises(capi.BisError):
        ctx.spmm(A, X, Y + 8, 4)                     # misaligned Y
    with pytest.raises(capi.BisError):
        ctx.call("bis_block_dot_to_slots", n, 9, X, Y, 120, None)   # slots 120 .. 128 past the bank
    with pytest.raises(capi.BisError):
        ctx.call("bis_block_cg_update", 0, n, 4, X, Y, X, Y, None, 40, 60, 126, 80, None)
    with pytest.raises(capi.BisError):
        ctx.call("bis_block_residual", 4, n, 4, X, Y, None, X, Y, None, 40, 60)    # sgs: not supported
    ctx.call("bis_block_dot_to_slots", n, 16, X, Y, 112, None)     # the last legal range
    ctx.set_option("factor_keep_crs", 0)
    try:
        L, U = ctx.split_triangular(A)
    finally:
        ctx.set_option("factor_keep_crs", 1)
    with pytest.raises(capi.BisError):
        ctx.spmm(L, X, Y, 4)                         # a factor without CRS arrays
    with pytest.raises(capi.BisError):
        host.solve_block(ctx, "sgs", crs=(rp, col, val), B=np.ones((n, 2)))
    L.free(), U.free(), A.free()
    ctx.free(X), ctx.free(Y)
    ctx.sync()


# ---- block CG ---------------------------------------------------------------------------------------------
def composition(ctx, A, n, b, x0, precond, max_iters, tol):
    """CG on one column through the existing single-vector entry points and the harness's stop rule."""
    pc = capi.PRECOND[precond]
    bb, xo, xn = ctx.upload(b), ctx.upload(x0), ctx.alloc(n)
    tmp, ro, rn, zo, zn, po, pn = (ctx.alloc(n) for _ in range(7))
    D = None
    if precond == "j":
        D = ctx.alloc(n)
        ctx.call("bis_matrix_extract_diagonal", A.h, D, None)
    ctx.call("bis_spmv", A.h, xo, tmp)
    ctx.call("bis_subtract_vectors", ro, bb, tmp, n, 1.0)
    if precond == "j":
        ctx.call("bis_elemwise_div_vectors", zo, ro, D, n, 1.0)
    else:
        ctx.call("bis_copy_vector", zo, ro, n)
    ctx.call("bis_copy_vector", po, zo, n)
    s_rz, s_rz_new = S_RZ, S_RZ_NEW
    ctx.call("bis_dot_to_slot", ro, zo, n, s_rz)
    ctx.call("bis_sumsq_to_slot", ro, n, S_RR)
    r0 = float(np.sqrt(ctx.scalars(S_RR)[0]))
    hist, it, thresh = [r0], 0, tol * r0
    while True:
        ctx.call("bis_spmv", A.h, po, tmp)
        ctx.call("bis_dot_to_slot", tmp, po, n, S_PAP)
        ctx.call("bis_cg_update", pc, n, None, xo, po, rn, ro, tmp, zn, D, s_rz, S_PAP, S_RR, s_rz_new)
        ctx.call("bis_cg_direction_x", n, pn, zn, po, xn, xo, s_rz_new, s_rz, S_PAP)
        it += 1
        nrm = float(np.sqrt(ctx.scalars(S_RR)[0]))
        hist.append(nrm)
        xo, xn, po, pn, ro, rn, zo, zn = xn, xo, pn, po, rn, ro, zn, zo
        s_rz, s_rz_new = s_rz_new, s_rz
        if nrm < thresh or it >= max_iters or nrm > np.finfo(float).max or np.isnan(nrm):
            break
    x = ctx.download(xo, n)
    for v in (bb, xo, xn, tmp, ro, rn, zo, zn, po, pn) + ((D,) if D else ()):
        ctx.free(v)
    return np.array(hist), it, bool(nrm < thresh), x


def block_case(n):
    """k = 8: ones, seeded random, an exact 2^-10 scaling of column 1, and a zero column started from x0 = 0."""
    rng = np.random.default_rng(7)
    B = rng.uniform(-1, 1, (n, 8))
    B[:, 0] = 1.0
    B[:, 4] = B[:, 1] * 2.0 ** -10
    B[:, 5] = 0.0
    X0 = np.full((n, 8), 0.1)
    X0[:, 4] = 0.1 * 2.0 ** -10
    X0[:, 5] = 0.0
    return B, X0


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


@pytest.mark.parametrize("precond", ["none", "j"])
@pytest.mark.parametrize("mat", ["hpcg32", "fdm2d16"])
def test_block_cg_vs_composition_bitwise(ctx, mat, precond):
    rp, col, val = named(mat)
    n = len(rp) - 1
    B, X0 = block_case(n)
    tol = 1e-8
    got = host.solve_block(ctx, precond, crs=(rp, col, val), B=B, X0=X0, tol=tol)
    A = ctx.upload_crs(rp, col, val)
    for j in range(8):
        hist, it, conv, x = composition(ctx, A, n, B[:, j].copy(), X0[:, j].copy(), precond, host.MAX_ITERS, tol)
        assert same(got.histories[j], hist), (mat, precond, j)
        assert got.iter_counts[j] == it and got.converged[j] == conv, (j, got.iter_counts[j], it)
        assert same(got.x_star[:, j], x), j
    A.free()
    # the zero column stops on its NaN at iteration 1 without disturbing the others
    assert got.iter_counts[5] == 1 and np.isnan(got.histories[5][1]) and not got.converged[5]
    assert all(got.converged[j] for j in range(8) if j != 5)
    its = set(int(v) for v in got.iter_counts)
    assert len(its) >= 2 and {v % 2 for v in its} == {0, 1}, its


@pytest.mark.parametrize("mat,k", [("hpcg32", 8), ("HPCG-128", 4)])
def test_block_cg_vs_single_rhs_and_oracle(ctx, mat, k):
    if mat == "hpcg32":
        rp, col, val = named(mat)
        kw = dict(crs=(rp, col, val))
    else:
        rp, col, val = matgen.hpcg(128)
        kw = dict(matrix_name=mat)
    n = len(rp) - 1
    B = np.random.default_rng(5).uniform(-1, 1, (n, k))
    B[:, 0] = 1.0
    X0 = np.full((n, k), 0.1)
    X0[:, -1] = np.random.default_rng(6).uniform(0, 1, n)
    tol = 1e-10
    got = host.solve_block(ctx, "none", B=B, X0=X0, tol=tol, **kw)
    for j in range(k):
        ref = port.solve(rp, col, val, "cg", "none", b=B[:, j], x0=X0[:, j], tol=tol)
        single = host.solve(ctx, "cg", "none", b=B[:, j], x0=X0[:, j], tol=tol, **kw)
        r0 = ref.history[0]
        for other in (ref, single):
            assert got.iter_counts[j] == other.iter_count, (j, got.iter_counts[j], other.iter_count)
            assert np.max(np.abs(got.histories[j] - other.history)) <= 1e-10 * r0, j
        assert got.converged[j]
        assert np.max(np.abs(got.x_star[:, j] - ref.x_star)) <= 1e-9 * np.max(np.abs(ref.x_star)), j
        assert abs(got.final_true_residuals[j] - ref.final_true_residual) <= 1e-10 * r0, j


def test_block_cg_invariance_bitwise(ctx):
    rp, col, val = named("hpcg32")
    n = len(rp) - 1
    B, X0 = block_case(n)
    crs = (rp, col, val)
    base = host.solve_block(ctx, "j", crs=crs, B=B, X0=X0, tol=1e-8)

    def eq(r, j, s, i):
        return (same(r.histories[j], s.histories[i]) and r.iter_counts[j] == s.iter_counts[i]
                and r.converged[j] == s.converged[i] and same(r.x_star[:, j], s.x_star[:, i]))

    # a column permutation of B permutes the results
    perm = np.array([3, 7, 0, 5, 1, 6, 2, 4])
    pr = host.solve_block(ctx, "j", crs=crs, B=B[:, perm], X0=X0[:, perm], tol=1e-8)
    assert all(eq(pr, i, base, perm[i]) for i in range(8))
    # column j of the k = 8 solve is the k = 1 solve of b_j
    for j in (0, 2, 5):
        one = host.solve_block(ctx, "j", crs=crs, B=B[:, j:j + 1], X0=X0[:, j:j + 1], tol=1e-8)
        assert eq(one, 0, base, j), j
    # graphs on and off, and a second run, give the same bits
    old = ctx.get_option("graph")
    try:
        ctx.set_option("graph", 1 - old)
        other = host.solve_block(ctx, "j", crs=crs, B=B, X0=X0, tol=1e-8)
    finally:
        ctx.set_option("graph", old)
    again = host.solve_block(ctx, "j", crs=crs, B=B, X0=X0, tol=1e-8)
    assert all(eq(other, j, base, j) and eq(again, j, base, j) for j in range(8))
    # a max_iters cap stops every running column there, as the composition does
    cap = host.solve_block(ctx, "j", crs=crs, B=B, X0=X0, tol=1e-8, max_iters=7)
    A = ctx.upload_crs(rp, col, val)
    for j in range(8):
        hist, it, conv, x = composition(ctx, A, n, B[:, j].copy(), X0[:, j].copy(), "j", 7, 1e-8)
        assert it == (1 if j == 5 else 7)
        assert same(cap.histories[j], hist) and cap.iter_counts[j] == it and same(cap.x_star[:, j], x), j
    A.free()


def test_block_cg_launches_and_profile_family(ctx):
    """The SpMM is counted in the "spmv" profile family; one block-CG iteration is 5 launches."""
    rp, col, val = named("hpcg16")
    n = len(rp) - 1
    A = ctx.upload_crs(rp, col, val)
    dX, dY = ctx.alloc(n * 4), ctx.alloc(n * 4)
    ctx.profile_enable(True)
    for _ in range(3):
        ctx.spmm(A, dX, dY, 4)
    ms, cnt = ctx.profile_read("spmv")
    ctx.profile_enable(False)
    assert cnt == 3 and ms > 0.0
    got = host.solve_block(ctx, "none", crs=(rp, col, val), B=np.ones((n, 3)), max_iters=10, tol=1e-30)
    assert list(got.iter_counts) == [10, 10, 10] and got.iterations == 10
    ctx.free(dX), ctx.free(dY), A.free()
