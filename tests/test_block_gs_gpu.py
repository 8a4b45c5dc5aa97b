"""GPU tests of multi-right-hand-side Gauss-Seidel and SGS (include/bis_b200.h, "multiple right-hand sides").

 - bis_block_sptrsv / bis_block_bsptrsv: every column bit-identical to the oracle's solve and to bis_sptrsv /
   bis_bsptrsv on that column; frozen columns untouched; the working arrays' clean/dirty tracking holds across
   single-vector solves and graph replays; errors are reported;
 - bis_spmm_sub: every column bit-identical to bis_spmv_sub;
 - host.solve_block(method="gs" | "sgs"): every column bit-identical to a Python composition of the single-vector
   entry points with the harness's stop rule, and x_star / iteration counts equal to the oracle's; invariant under
   column permutation, k, graphs and a max_iters cap; launch counts, profile family and device memory.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import golden
from oracle import matgen, port

from basic_iterative_solvers_b200 import capi, host

pytestmark = pytest.mark.gpu

S_RR = 0


def named(name):
    if name == "hpcg16":
        return matgen.hpcg(16)
    if name == "hpcg32":
        return matgen.hpcg(32)
    g = golden(name)
    return g["rp"], g["col"], g["val"]


def long_rows(n, seed):
    """Nonsymmetric, diagonally dominant, columns ascending; rows of both factors up to 40 nonzeros (more than the
    block solve's register window of 8 or 16)."""
    rng = np.random.default_rng(seed)
    rows, vals = [], []
    for i in range(n):
        m = int(rng.integers(0, 41)) if i % 5 else 0
        c = np.unique(np.concatenate([rng.choice(n, size=min(m, n), replace=False), [i]])).astype(np.int32)
        v = rng.uniform(-1, 1, c.size)
        v[c == i] = 50.0 + rng.uniform(0, 1)
        rows.append(c)
        vals.append(v)
    rp = np.zeros(n + 1, np.int32)
    rp[1:] = np.cumsum([len(r) for r in rows])
    return rp, np.concatenate(rows), np.concatenate(vals)


MATRICES = {
    "hpcg16": lambda: named("hpcg16"),
    "hpcg32": lambda: named("hpcg32"),
    "fdm2d16": lambda: named("fdm2d16"),
    "band_klein": lambda: named("band_klein"),
    "random300": lambda: named("random300"),
    "anderson": lambda: named("anderson_12_10_8"),
    "long_rows": lambda: long_rows(600, 9),
    "hpcg16_rp64": lambda: tuple([named("hpcg16")[0].astype(np.int64)] + list(named("hpcg16")[1:])),
}


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


class Factors:
    """A on the device, its strict factors (CRS kept), A's diagonal on the device and the host CRS of the factors."""

    def __init__(self, ctx, rp, col, val):
        self.ctx = ctx
        self.n = len(rp) - 1
        self.A = ctx.upload_crs(rp, col, val)
        self.L, self.U = ctx.split_triangular(self.A)
        self.dD = ctx.alloc(self.n)
        ctx.call("bis_matrix_extract_diagonal", self.A.h, self.dD, None)
        self.D = ctx.download(self.dD, self.n)
        self.Lh = self.L.download()
        self.Uh = self.U.download()

    def free(self):
        self.ctx.free(self.dD)
        self.L.free(), self.U.free(), self.A.free()


def block_solve(ctx, f, T, k, B, X0=None, active=None, backward=False, alias=False):
    n = f.n
    dB = ctx.upload(B)
    dX = dB if alias else ctx.upload(np.full((n, k), np.nan) if X0 is None else X0)
    dA = None if active is None else ctx.upload(np.asarray(active, np.float64))
    ctx.call("bis_block_bsptrsv" if backward else "bis_block_sptrsv", T.h, k, dX, f.dD, dB, dA)
    X = ctx.download(dX, n * k).reshape(n, k)
    ctx.free(dB)
    if not alias:
        ctx.free(dX)
    if dA is not None:
        ctx.free(dA)
    return X


def single_solve(ctx, f, T, b, backward=False):
    db, dx = ctx.upload(b), ctx.alloc(f.n)
    ctx.call("bis_bsptrsv" if backward else "bis_sptrsv", T.h, dx, f.dD, db)
    x = ctx.download(dx, f.n)
    ctx.free(db), ctx.free(dx)
    return x


# ---- kernels -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 2, 3, 5, 8, 16])
@pytest.mark.parametrize("mat", list(MATRICES))
def test_block_sptrsv_vs_oracle_and_single_bitwise(ctx, mat, k):
    rp, col, val = MATRICES[mat]()
    f = Factors(ctx, rp, col, val)
    if mat.endswith("rp64"):
        assert f.A.info()["rp_bytes"] == 8
    B = np.random.default_rng(k).uniform(-1, 1, (f.n, k))
    for backward, T, Th in ((False, f.L, f.Lh), (True, f.U, f.Uh)):
        X = block_solve(ctx, f, T, k, B, backward=backward)
        for j in range(k):
            ref = port.sptrsv(Th[0], Th[1], Th[2], f.D, B[:, j].copy(), backward=backward)
            assert same(X[:, j], ref), (mat, k, backward, j)
            assert same(X[:, j], single_solve(ctx, f, T, B[:, j].copy(), backward)), (mat, k, backward, j)
    f.free()


@pytest.mark.parametrize("k", [3, 16])
def test_block_sptrsv_alias_and_released_crs_bitwise(ctx, k):
    rp, col, val = named("hpcg32")
    f = Factors(ctx, rp, col, val)
    B = np.random.default_rng(3).uniform(-1, 1, (f.n, k))
    want_l = np.stack([port.sptrsv(*f.Lh, f.D, B[:, j].copy()) for j in range(k)], axis=1)
    want_u = np.stack([port.sptrsv(*f.Uh, f.D, B[:, j].copy(), backward=True) for j in range(k)], axis=1)
    # X aliasing B
    assert same(block_solve(ctx, f, f.L, k, B, alias=True), want_l)
    assert same(block_solve(ctx, f, f.U, k, B, alias=True, backward=True), want_u)
    # factors that gave up their natural-order CRS
    ctx.set_option("factor_keep_crs", 0)
    try:
        L2, U2 = ctx.split_triangular(f.A)
    finally:
        ctx.set_option("factor_keep_crs", 1)
    assert same(block_solve(ctx, f, L2, k, B), want_l)
    assert same(block_solve(ctx, f, U2, k, B, backward=True), want_u)
    L2.free(), U2.free()
    f.free()


def test_block_sptrsv_beside_wavefront_hpcg64_bitwise(ctx):
    """The single-vector solve forced onto the stencil wavefront; the block solve ignores trsv_variant."""
    rp, col, val = matgen.hpcg(64)
    ctx.set_option("trsv_variant", 5)
    try:
        f = Factors(ctx, rp, col, val)
        k = 5
        B = np.random.default_rng(4).uniform(-1, 1, (f.n, k))
        for backward, T in ((False, f.L), (True, f.U)):
            X = block_solve(ctx, f, T, k, B, backward=backward)
            w0 = ctx.info()["wave_solves"]
            for j in range(k):
                assert same(X[:, j], single_solve(ctx, f, T, B[:, j].copy(), backward)), (backward, j)
            assert ctx.info()["wave_solves"] - w0 == k
            Th = f.Uh if backward else f.Lh
            assert same(X[:, 2], port.sptrsv(*Th, f.D, B[:, 2].copy(), backward=backward))
        f.free()
    finally:
        ctx.set_option("trsv_variant", 0)


@pytest.mark.parametrize("k", [2, 5, 16])
def test_block_sptrsv_frozen_columns_bitwise(ctx, k):
    rp, col, val = named("fdm2d16")
    f = Factors(ctx, rp, col, val)
    B = np.random.default_rng(k + 1).uniform(-1, 1, (f.n, k))
    active = np.ones(k)
    active[::2] = 0.0
    fill = np.full((f.n, k), np.nan)
    for backward, T in ((False, f.L), (True, f.U)):
        full = block_solve(ctx, f, T, k, B, backward=backward, active=None)
        part = block_solve(ctx, f, T, k, B, X0=fill, backward=backward, active=active)
        for j in range(k):
            if active[j]:
                assert same(part[:, j], full[:, j]), (backward, j)
            else:
                assert np.array_equal(bits(part[:, j].copy()), bits(fill[:, j].copy())), (backward, j)
    f.free()


def test_block_sptrsv_interleaved_and_after_graph_bitwise(ctx):
    """Single-vector and block solves alternated on one factor, block solves of different k, and block solves after
    graph replays of a block solve, all give the same bits (the working arrays are tracked as clean or dirty)."""
    rp, col, val = named("hpcg32")
    f = Factors(ctx, rp, col, val)
    n = f.n
    B = np.random.default_rng(8).uniform(-1, 1, (n, 8))
    want = block_solve(ctx, f, f.L, 8, B)
    for j in range(8):
        assert same(single_solve(ctx, f, f.L, B[:, j].copy()), want[:, j])
        assert same(block_solve(ctx, f, f.L, 8, B), want)
        assert same(block_solve(ctx, f, f.L, 3, B[:, :3].copy()), want[:, :3])
    dB, dX = ctx.upload(B), ctx.alloc(n * 8)
    ctx.call("bis_graph_begin")
    ctx.call("bis_block_sptrsv", f.L.h, 8, dX, f.dD, dB, None)
    g = C.c_void_p()
    ctx.call("bis_graph_end", C.byref(g))
    for _ in range(3):
        ctx.call("bis_init_vector", dX, 0.0, n * 8)
        ctx.call("bis_graph_launch", g)
        assert same(ctx.download(dX, n * 8).reshape(n, 8), want)
        assert same(block_solve(ctx, f, f.L, 8, B), want)
        assert same(single_solve(ctx, f, f.L, B[:, 1].copy()), want[:, 1])
    ctx.call("bis_graph_free", g)
    ctx.free(dB), ctx.free(dX)
    f.free()


@pytest.mark.parametrize("k", [1, 3, 8, 16])
@pytest.mark.parametrize("mat", ["hpcg32", "random300", "long_rows"])
def test_spmm_sub_vs_spmv_sub_bitwise(ctx, mat, k):
    rp, col, val = MATRICES[mat]()
    f = Factors(ctx, rp, col, val)
    n = f.n
    rng = np.random.default_rng(k)
    X, B = rng.uniform(-1, 1, (n, k)), rng.uniform(-1, 1, (n, k))
    dX, dB, dY = ctx.upload(X), ctx.upload(B), ctx.alloc(n * k)
    dx, db, dy = ctx.alloc(n), ctx.alloc(n), ctx.alloc(n)
    for T in (f.L, f.U):
        ctx.call("bis_init_vector", dY, np.nan, n * k)
        ctx.call("bis_spmm_sub", T.h, k, dX, dB, dY)
        Y = ctx.download(dY, n * k).reshape(n, k)
        for j in range(k):
            ctx.upload(X[:, j].copy(), dx)
            ctx.upload(B[:, j].copy(), db)
            ctx.call("bis_spmv_sub", T.h, dx, db, dy)
            assert same(Y[:, j], ctx.download(dy, n)), (mat, k, j)
    for v in (dX, dB, dY, dx, db, dy):
        ctx.free(v)
    f.free()


def test_block_gs_entry_points_fail_loudly(ctx):
    rp, col, val = named("hpcg16")
    f = Factors(ctx, rp, col, val)
    n = f.n
    X, B = ctx.alloc(n * 17 + 2), ctx.alloc(n * 17 + 2)
    ctx.call("bis_init_vector", X, 0.0, n * 17 + 2)
    ctx.call("bis_init_vector", B, 1.0, n * 17 + 2)
    for name, T in (("bis_block_sptrsv", f.L), ("bis_block_bsptrsv", f.U)):
        for k in (0, 17):
            with pytest.raises(capi.BisError):
                ctx.call(name, T.h, k, X, f.dD, B, None)
        with pytest.raises(capi.BisError):
            ctx.call(name, T.h, 4, X + 8, f.dD, B, None)      # misaligned X
        with pytest.raises(capi.BisError):
            ctx.call(name, T.h, 4, X, f.dD, B + 8, None)      # misaligned B
        with pytest.raises(capi.BisError):
            ctx.call(name, T.h, 4, X, None, B, None)          # null D
    with pytest.raises(capi.BisError):
        ctx.call("bis_block_sptrsv", f.U.h, 4, X, f.dD, B, None)   # the wrong triangle
    with pytest.raises(capi.BisError):
        ctx.call("bis_block_bsptrsv", f.L.h, 4, X, f.dD, B, None)
    with pytest.raises(capi.BisError):
        ctx.call("bis_block_sptrsv", f.A.h, 4, X, f.dD, B, None)   # not triangular
    for k in (0, 17):
        with pytest.raises(capi.BisError):
            ctx.call("bis_spmm_sub", f.L.h, k, X, B, X + 16 * n * 8)
    with pytest.raises(capi.BisError):
        ctx.call("bis_spmm_sub", f.L.h, 4, X, B + 8, X + 16 * n * 8)   # misaligned B
    ctx.call("bis_block_sptrsv", f.L.h, 16, X, f.dD, B, None)           # the largest legal k
    ctx.free(X), ctx.free(B)
    f.free()
    ctx.sync()


# ---- block GS / SGS ----------------------------------------------------------------------------------------------
def composition(ctx, A, L, U, dD, n, b, x0, sgs, max_iters, tol):
    """GS / SGS on one column through the single-vector entry points and the harness's stop rule."""
    bb, x, tmp, ax, r = ctx.upload(b), ctx.upload(x0), ctx.alloc(n), ctx.alloc(n), ctx.alloc(n)

    def norm():
        ctx.call("bis_spmv", A.h, x, ax)
        ctx.call("bis_subtract_vectors", r, bb, ax, n, 1.0)
        ctx.call("bis_sumsq_to_slot", r, n, S_RR)
        return float(np.sqrt(ctx.scalars(S_RR)[0]))

    r0 = norm()
    hist, it, thresh = [r0], 0, tol * r0
    while True:
        ctx.call("bis_spmv_sub", U.h, x, bb, tmp)
        ctx.call("bis_sptrsv", L.h, x, dD, tmp)
        if sgs:
            ctx.call("bis_spmv_sub", L.h, x, bb, tmp)
            ctx.call("bis_bsptrsv", U.h, x, dD, tmp)
        it += 1
        nrm = norm()
        hist.append(nrm)
        if nrm < thresh or it >= max_iters or nrm > np.finfo(float).max or np.isnan(nrm):
            break
    xs = ctx.download(x, n)
    for v in (bb, x, tmp, ax, r):
        ctx.free(v)
    return np.array(hist), it, bool(nrm < thresh), xs


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


def check_vs_composition(ctx, got, rp, col, val, B, X0, sgs, max_iters, tol):
    f = Factors(ctx, rp, col, val)
    for j in range(B.shape[1]):
        hist, it, conv, x = composition(ctx, f.A, f.L, f.U, f.dD, f.n, B[:, j].copy(), X0[:, j].copy(), sgs,
                                        max_iters, tol)
        assert same(got.histories[j], hist), j
        assert got.iter_counts[j] == it and got.converged[j] == conv, (j, got.iter_counts[j], it)
        assert same(got.x_star[:, j], x), j
    f.free()


@pytest.mark.parametrize("method", ["gs", "sgs"])
@pytest.mark.parametrize("mat", ["hpcg32", "fdm2d16"])
def test_block_gs_vs_composition_bitwise(ctx, mat, method):
    rp, col, val = named(mat)
    n = len(rp) - 1
    B, X0 = block_case(n)
    tol, cap = 1e-8, host.MAX_ITERS
    got = host.solve_block(ctx, "none", crs=(rp, col, val), B=B, X0=X0, tol=tol, max_iters=cap, method=method)
    check_vs_composition(ctx, got, rp, col, val, B, X0, method == "sgs", cap, tol)
    # the zero column: its residual stays 0, never below a threshold of 0, so it runs to the cap; the others
    # converge, at different iterations
    assert got.iter_counts[5] == cap and not got.converged[5] and not np.any(got.histories[5])
    assert all(got.converged[j] for j in range(8) if j != 5)
    assert len(set(int(got.iter_counts[j]) for j in range(8) if j != 5)) >= 2, got.iter_counts


@pytest.mark.parametrize("method", ["gs", "sgs"])
@pytest.mark.parametrize("mat,k", [("hpcg32", 8), ("HPCG-128", 4)])
def test_block_gs_vs_single_rhs_and_oracle(ctx, mat, k, method):
    """hpcg32: a real solve (tol 1e-8; the slow columns of GS reach MAX_ITERS).  HPCG-128 (device generation):
    60 iterations, which keeps the oracle's CPU sweeps short."""
    if mat == "hpcg32":
        rp, col, val = named(mat)
        kw = dict(crs=(rp, col, val), tol=1e-8)
    else:
        rp, col, val = matgen.hpcg(128)
        kw = dict(matrix_name=mat, tol=1e-10, max_iters=60)
    n = len(rp) - 1
    B = np.random.default_rng(5).uniform(-1, 1, (n, k))
    B[:, 0] = 1.0
    X0 = np.full((n, k), 0.1)
    X0[:, -1] = np.random.default_rng(6).uniform(0, 1, n)
    got = host.solve_block(ctx, "none", B=B, X0=X0, method=method, **kw)
    for j in range(k):
        ref = port.solve(rp, col, val, method, "none", b=B[:, j], x0=X0[:, j], tol=kw["tol"],
                         max_iters=kw.get("max_iters", 0))
        single = host.solve(ctx, method, "none", b=B[:, j], x0=X0[:, j], **kw)
        r0 = ref.history[0]
        assert got.iter_counts[j] == ref.iter_count == single.iter_count, (j, got.iter_counts[j], ref.iter_count)
        assert got.converged[j] == ref.converged == single.converged, j
        assert same(got.x_star[:, j], ref.x_star), j
        for other in (ref, single):
            assert np.max(np.abs(got.histories[j] - other.history)) <= 1e-10 * r0, j
        assert abs(got.final_true_residuals[j] - ref.final_true_residual) <= 1e-10 * r0, j
    if mat == "hpcg32":
        assert any(got.converged), got.iter_counts


@pytest.mark.parametrize("method", ["gs", "sgs"])
def test_block_gs_invariance_bitwise(ctx, method):
    rp, col, val = named("hpcg32")
    n = len(rp) - 1
    B, X0 = block_case(n)
    crs = (rp, col, val)
    kw = dict(crs=crs, tol=1e-8, max_iters=100, method=method)
    base = host.solve_block(ctx, "none", B=B, X0=X0, **kw)

    def eq(r, j, s, i):
        return (same(r.histories[j], s.histories[i]) and r.iter_counts[j] == s.iter_counts[i]
                and r.converged[j] == s.converged[i] and same(r.x_star[:, j], s.x_star[:, i]))

    perm = np.array([3, 7, 0, 5, 1, 6, 2, 4])
    pr = host.solve_block(ctx, "none", B=B[:, perm], X0=X0[:, perm], **kw)
    assert all(eq(pr, i, base, perm[i]) for i in range(8))
    for j in (0, 2, 5):
        one = host.solve_block(ctx, "none", B=B[:, j:j + 1], X0=X0[:, j:j + 1], **kw)
        assert eq(one, 0, base, j), j
    old = ctx.get_option("graph")
    try:
        ctx.set_option("graph", 1 - old)
        other = host.solve_block(ctx, "none", B=B, X0=X0, **kw)
    finally:
        ctx.set_option("graph", old)
    again = host.solve_block(ctx, "none", B=B, X0=X0, **kw)
    assert all(eq(other, j, base, j) and eq(again, j, base, j) for j in range(8))
    cap = host.solve_block(ctx, "none", B=B, X0=X0, **dict(kw, max_iters=7))
    assert list(cap.iter_counts) == [7] * 8
    check_vs_composition(ctx, cap, rp, col, val, B, X0, method == "sgs", 7, 1e-8)


# ---- shape ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("method,per_iter,solves", [("gs", 5, 1), ("sgs", 7, 2)])
def test_block_gs_launches_profile_and_memory(ctx, method, per_iter, solves):
    rp, col, val = named("hpcg32")
    n = len(rp) - 1
    kw = dict(crs=(rp, col, val), B=np.ones((n, 3)), X0=np.full((n, 3), 0.1), tol=1e-30, method=method)
    old = ctx.get_option("graph")
    try:
        # status, the SpMM forms, the block solves and the residual; the working arrays stay clean from solve to solve
        ctx.set_option("graph", 0)
        a = host.solve_block(ctx, "none", **kw, max_iters=10)
        b = host.solve_block(ctx, "none", **kw, max_iters=20)
        assert list(b.iter_counts) == [20] * 3 and b.iterations == 20
        assert b.launches - a.launches == 10 * per_iter, (a.launches, b.launches)
        # in a graph the tracking cannot know which array a replay left clean: one sentinel fill per block solve
        ctx.set_option("graph", 1)
        a = host.solve_block(ctx, "none", **kw, max_iters=10)
        b = host.solve_block(ctx, "none", **kw, max_iters=20)
        assert b.launches - a.launches == 10 * (per_iter + solves), (a.launches, b.launches)
    finally:
        ctx.set_option("graph", old)
    # the block solves count in "sptrsv", the SpMM forms in "spmv"
    f = Factors(ctx, rp, col, val)
    dX, dB, dT = ctx.upload(np.ones((n, 4))), ctx.upload(np.ones((n, 4))), ctx.alloc(n * 4)
    ctx.profile_enable(True)
    try:
        ctx.call("bis_block_sptrsv", f.L.h, 4, dX, f.dD, dB, None)
        ctx.call("bis_block_bsptrsv", f.U.h, 4, dX, f.dD, dB, None)
        ms, cnt = ctx.profile_read("sptrsv")
        ctx.call("bis_spmm_sub", f.U.h, 4, dX, dB, dT)
        _, cnt_spmv = ctx.profile_read("spmv")
    finally:
        ctx.profile_enable(False)
    assert cnt == 2 and ms > 0.0 and cnt_spmv == 1
    ctx.free(dX), ctx.free(dB), ctx.free(dT)
    f.free()
    # freeing a factor returns its working arrays (2 x n x 16 doubles here)
    rp, col, val = matgen.hpcg(64)
    cache = ctx.get_option("vector_cache")
    ctx.set_option("vector_cache", 0)
    try:
        f = Factors(ctx, rp, col, val)
        dX = ctx.upload(np.ones((f.n, 16)))
        ctx.sync()
        free0 = ctx.info()["free"]
        ctx.call("bis_block_sptrsv", f.L.h, 16, dX, f.dD, dX, None)
        ctx.sync()
        free1 = ctx.info()["free"]
        ctx.free(dX)
        f.L.free()
        ctx.sync()
        free2 = ctx.info()["free"]
        f.free()
    finally:
        ctx.set_option("vector_cache", cache)
    arrays = 2 * f.n * 16 * 8
    assert free0 - free1 >= arrays, (free0, free1, arrays)
    # L's level sets and copy plus the arrays come back (and dX)
    assert free2 - free1 >= arrays + f.n * 16 * 8, (free1, free2)


def test_block_gs_rejections(ctx):
    rp, col, val = named("hpcg16")
    n = len(rp) - 1
    B = np.ones((n, 2))
    with pytest.raises(capi.BisError):
        host.solve_block(ctx, "j", crs=(rp, col, val), B=B, method="gs")
    with pytest.raises(capi.BisError):
        host.solve_block(ctx, "sgs", crs=(rp, col, val), B=B, method="sgs")
    ctx.set_option("perm_mode", 2)
    try:
        with pytest.raises(capi.BisError):
            host.solve_block(ctx, "none", crs=(rp, col, val), B=B, method="gs")
    finally:
        ctx.set_option("perm_mode", 0)
    with pytest.raises(capi.BisError):
        host.solve_block(ctx, "none", crs=(rp, col, val), B=np.ones((n, 17)), method="sgs")
    with pytest.raises(ValueError):
        host.solve_block(ctx, "none", crs=(rp, col, val), B=B, method="j")
