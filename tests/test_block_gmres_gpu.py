"""GPU tests of the multi-right-hand-side GMRES (include/bis_b200.h, "Block GMRES"; host/methods/block_gmres.hpp).

 - the batched GMRES kernels: every column bit-identical to the single-vector entry point it batches, frozen columns
   untouched, and the split vector read equal to bis_vector_download;
 - the entry points and solve_block(method="gm") fail loudly on bad arguments;
 - block GMRES: every column bit-identical to a per-column composition of the single-vector entry points with the
   harness's stop and restart rules (a Python loop below); within the north-star bar of host.solve("gm") and of the
   oracle; invariant under column permutation, k, graphs and a max_iters cap; launches, profile family and memory.
"""
import ctypes as C
import math

import numpy as np
import pytest

from conftest import golden
from oracle import matgen, port

from basic_iterative_solvers_b200 import capi, host

pytestmark = pytest.mark.gpu

NAN = float("nan")
JACOBI = capi.PRECOND["j"]
S_RR, S_BETA2, S_H, S_TMP = 0, 10, 16, 100


def named(name):
    if name == "hpcg32":
        return matgen.hpcg(32)
    g = golden(name)
    return g["rp"], g["col"], g["val"]


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture
def no_vector_cache(ctx):
    old = ctx.get_option("vector_cache")
    ctx.set_option("vector_cache", 0)
    yield
    ctx.set_option("vector_cache", old)


# ---- kernels -----------------------------------------------------------------------------------------------
def stride(n, k):
    return n * k + (n * k) % 2


def blocks(ctx, rng, n, k, nblk, ldv):
    """nblk random n x k blocks at V + l*ldv (host copy [nblk, n, k]); the pad element of an odd n*k is NaN."""
    host_v = rng.uniform(-1, 1, (nblk, n, k))
    flat = np.full(nblk * ldv, NAN)
    for l in range(nblk):
        flat[l * ldv:l * ldv + n * k] = host_v[l].ravel()
    return ctx.upload(flat), host_v


def active_flags(k):
    return np.array([0.0 if (k > 1 and j % 3 == 1) else 1.0 for j in range(k)])


def single(ctx, v):
    return ctx.upload(np.ascontiguousarray(v))


KERNEL_CASES = [(n, k) for k in (1, 3, 8, 16) for n in (1001, 2048)]


@pytest.mark.parametrize("n,k", KERNEL_CASES)
@pytest.mark.parametrize("precond", ["none", "j"])
def test_precond_dot_bitwise(ctx, n, k, precond):
    rng = np.random.default_rng(100 * k + n % 7)
    ldv = stride(n, k)
    V, Vh = blocks(ctx, rng, n, k, 2, ldv)
    W0 = rng.uniform(-1, 1, (n, k))
    d = rng.uniform(0.5, 2.0, n)
    dW, dD = ctx.upload(W0), ctx.upload(d)
    act = active_flags(k)
    dact = ctx.upload(act)
    H = ctx.upload(np.full(6 * k, NAN))
    for v0 in (V, None):   # (W, V0) and, without V0, (W, W)
        ctx.upload(W0, dW)
        ctx.upload(np.full(6 * k, NAN), H)
        ctx.call("bis_block_gmres_precond_dot", capi.PRECOND[precond], n, k, dW, dD, v0, H, dact)
        W = ctx.download(dW, n * k).reshape(n, k)
        h = ctx.download(H, 6 * k)
        w1, vv, dd = ctx.alloc(n), single(ctx, Vh[0][:, 0]), single(ctx, d)
        for j in range(k):
            ctx.upload(W0[:, j].copy(), w1)
            ctx.upload(Vh[0][:, j].copy(), vv)
            if precond == "j":
                ctx.call("bis_elemwise_div_vectors", w1, w1, dd, n, 1.0)
            ctx.call("bis_dot_to_slot", w1, vv if v0 else w1, n, S_TMP)
            if act[j]:
                assert same(W[:, j], ctx.download(w1, n)), j
                assert same(h[j], ctx.scalars(S_TMP)[0]), j
            else:
                assert same(W[:, j], W0[:, j]) and np.isnan(h[j]), j
        assert np.all(np.isnan(h[k:]))
        for p in (w1, vv, dd):
            ctx.free(p)
    for p in (V, dW, dD, dact, H):
        ctx.free(p)


@pytest.mark.parametrize("n,k", KERNEL_CASES)
def test_mgs_step_and_scale_bitwise(ctx, n, k):
    rng = np.random.default_rng(200 * k + n % 5)
    ldv = stride(n, k)
    V, Vh = blocks(ctx, rng, n, k, 4, ldv)
    W0 = rng.uniform(-1, 1, (n, k))
    dW = ctx.upload(W0)
    act = active_flags(k)
    dact = ctx.upload(act)
    w1, vl, vn, out1 = (ctx.alloc(n) for _ in range(4))
    for l, with_next in ((0, True), (2, True), (2, False)):
        Hh = np.full(6 * k, NAN)
        Hh[l * k:(l + 1) * k] = rng.uniform(-0.5, 0.5, k)
        H = ctx.upload(Hh)
        ctx.upload(W0, dW)
        vnext = V + 8 * (l + 1) * ldv if with_next else None
        ctx.call("bis_block_mgs_step", n, k, dW, V + 8 * l * ldv, vnext, H, l, dact)
        W = ctx.download(dW, n * k).reshape(n, k)
        h = ctx.download(H, 6 * k)
        for j in range(k):
            ctx.upload(W0[:, j].copy(), w1)
            ctx.upload(Vh[l][:, j].copy(), vl)
            ctx.upload(Vh[l + 1][:, j].copy(), vn)
            ctx.call("bis_scalar_set", S_TMP, float(Hh[l * k + j]))
            ctx.call("bis_mgs_step", n, w1, vl, vn if with_next else None, S_TMP, S_TMP + 1)
            if act[j]:
                assert same(W[:, j], ctx.download(w1, n)), (l, j)
                assert same(h[(l + 1) * k + j], ctx.scalars(S_TMP + 1)[0]), (l, j)
            else:
                assert same(W[:, j], W0[:, j]) and np.isnan(h[(l + 1) * k + j]), (l, j)
        assert same(h[l * k:(l + 1) * k], Hh[l * k:(l + 1) * k])
        ctx.free(H)
    # scale: out = W * (1 / sqrt(H[l, j])) into a NaN-filled block
    l = 3
    Hh = np.full(6 * k, NAN)
    Hh[l * k:(l + 1) * k] = rng.uniform(0.1, 4.0, k)
    H = ctx.upload(Hh)
    ctx.upload(W0, dW)
    out = ctx.upload(np.full(n * k, NAN))
    ctx.call("bis_block_scale_inv_norm", n, k, out, dW, H, l, dact)
    got = ctx.download(out, n * k).reshape(n, k)
    for j in range(k):
        ctx.upload(W0[:, j].copy(), w1)
        ctx.call("bis_scalar_set", S_TMP, float(Hh[l * k + j]))
        ctx.call("bis_scale_inv_norm", n, out1, w1, S_TMP)
        want = ctx.download(out1, n) if act[j] else np.full(n, NAN)
        assert same(got[:, j], want), j
    assert same(ctx.download(H, 6 * k), Hh)
    for p in (V, dW, dact, w1, vl, vn, out1, H, out):
        ctx.free(p)


@pytest.mark.parametrize("n,k", KERNEL_CASES)
def test_update_x_bitwise(ctx, n, k):
    rng = np.random.default_rng(300 * k + n % 3)
    ldv = stride(n, k)
    nbmax = 5
    V, Vh = blocks(ctx, rng, n, k, nbmax + 1, ldv)
    Xo = rng.uniform(-1, 1, (n, k))
    dXo = ctx.upload(Xo)
    mask = np.array([1 if j % 3 != 1 or k == 1 else 0 for j in range(k)], np.int32)
    x1, xo1 = ctx.alloc(n), ctx.alloc(n)
    Vs = ctx.alloc(nbmax * n)
    for nb in (0, 1, nbmax):
        Y = rng.uniform(-2, 2, (k, max(nb, 1)))[:, :nb].copy()
        dX = ctx.upload(np.full(n * k, NAN))
        ctx.call("bis_block_gmres_update_x", n, k, nb, V, ldv, ptr(Y), dX, dXo, ptr(mask))
        X = ctx.download(dX, n * k).reshape(n, k)
        for j in range(k):
            if not mask[j]:
                assert np.all(np.isnan(X[:, j])), (nb, j)
                continue
            ctx.upload(np.concatenate([Vh[l][:, j] for l in range(nbmax)]), Vs)
            ctx.upload(Xo[:, j].copy(), xo1)
            y = np.ascontiguousarray(Y[j]) if nb else np.zeros(1)
            ctx.call("bis_gmres_update_x", n, nb, Vs, ptr(y), x1, xo1, None)
            assert same(X[:, j], ctx.download(x1, n)), (nb, j)
        # in place (X == X_old), as the block solver runs it
        ctx.upload(Xo, dX)
        ctx.call("bis_block_gmres_update_x", n, k, nb, V, ldv, ptr(Y), dX, dX, ptr(mask))
        Xi = ctx.download(dX, n * k).reshape(n, k)
        assert same(Xi[:, mask == 1], X[:, mask == 1]) and same(Xi[:, mask == 0], Xo[:, mask == 0])
        ctx.free(dX)
    for p in (V, dXo, x1, xo1, Vs):
        ctx.free(p)


def test_vector_read_matches_download(ctx):
    vals = np.random.default_rng(1).uniform(-1, 1, 1056)
    d = ctx.upload(vals)
    for off, cnt in ((0, 1056), (3, 17), (0, 1)):
        ctx.call("bis_vector_read_begin", d + 8 * off, cnt)
        ctx.call("bis_scalar_read_begin", S_RR, 2)   # a scalar read may be outstanding at the same time
        out = np.zeros(cnt)
        ctx.call("bis_vector_read_end", ptr(out), cnt)
        ctx.call("bis_scalar_read_end", S_RR, 2, (C.c_double * 2)())
        assert same(out, ctx.download(d + 8 * off, cnt)) and same(out, vals[off:off + cnt])
    with pytest.raises(capi.BisError):
        ctx.call("bis_vector_read_begin", d, 4097)   # past BIS_VECTOR_READ_MAX
    with pytest.raises(capi.BisError):
        ctx.call("bis_vector_read_begin", d, 0)
    ctx.free(d)


def test_block_gmres_entry_points_fail_loudly(ctx):
    rp, col, val = named("hpcg32")
    n = 1001
    X, Y = ctx.alloc(n * 17 + 2), ctx.alloc(n * 17 + 2)
    H = ctx.alloc(66 * 17)
    y = np.zeros(17 * 4)
    mask = np.ones(17, np.int32)
    for k in (0, 17):
        for call in (("bis_block_gmres_precond_dot", 0, n, k, X, None, Y, H, None),
                     ("bis_block_mgs_step", n, k, X, Y, None, H, 0, None),
                     ("bis_block_scale_inv_norm", n, k, Y, X, H, 0, None),
                     ("bis_block_gmres_update_x", n, k, 2, Y, n * max(k, 1) + 1, ptr(y), X, X, ptr(mask))):
            with pytest.raises(capi.BisError):
                ctx.call(*call)
    bad = (("bis_block_gmres_precond_dot", 0, n, 3, X + 8, None, Y, H, None),     # misaligned W
           ("bis_block_gmres_precond_dot", 0, n, 3, X, None, Y + 8, H, None),     # misaligned V0
           ("bis_block_mgs_step", n, 3, X, Y + 8, None, H, 0, None),              # misaligned V_l
           ("bis_block_scale_inv_norm", n, 3, Y + 8, X, H, 0, None),              # misaligned out
           ("bis_block_gmres_update_x", n, 3, 2, Y + 8, 3004, ptr(y), X, X, ptr(mask)),   # misaligned V
           ("bis_block_gmres_update_x", n, 3, 2, Y, 3003, ptr(y), X, X, ptr(mask)),       # odd ldv
           ("bis_block_gmres_update_x", n, 3, 2, Y, 3002, ptr(y), X, X, ptr(mask)),       # ldv < n*k
           ("bis_block_gmres_update_x", n, 3, 65, Y, 3004, ptr(y), X, X, ptr(mask)),      # nb > 64
           ("bis_block_mgs_step", n, 3, X, Y, None, H, -1, None),                 # l out of range
           ("bis_block_mgs_step", n, 3, X, Y, None, H, 64, None),
           ("bis_block_scale_inv_norm", n, 3, Y, X, H, -1, None),
           ("bis_block_scale_inv_norm", n, 3, Y, X, H, 65, None),
           ("bis_block_gmres_precond_dot", 0, n, 3, X, None, Y, None, None),      # null H
           ("bis_block_mgs_step", n, 3, X, Y, None, None, 0, None),
           ("bis_block_scale_inv_norm", n, 3, Y, X, None, 0, None),
           ("bis_block_gmres_precond_dot", capi.PRECOND["gs"], n, 3, X, Y, Y, H, None),   # gs: not supported
           ("bis_block_gmres_precond_dot", JACOBI, n, 3, X, None, Y, H, None))    # jacobi without a diagonal
    for call in bad:
        with pytest.raises(capi.BisError):
            ctx.call(*call)
    ctx.call("bis_block_mgs_step", n, 3, X, Y, None, H, 63, None)              # the last legal rows
    ctx.call("bis_block_scale_inv_norm", n, 3, Y, X, H, 64, None)
    for p in (X, Y, H):
        ctx.free(p)
    ctx.sync()
    B = np.ones((len(rp) - 1, 2))
    for kw in (dict(precond="sgs"), dict(precond="ilu0"), dict(restart_len=0), dict(restart_len=65)):
        with pytest.raises(capi.BisError):
            host.solve_block(ctx, kw.pop("precond", "none"), crs=(rp, col, val), B=B, method="gm", **kw)
    with pytest.raises(ValueError):
        host.solve_block(ctx, "none", crs=(rp, col, val), B=B, method="bi")
    old = ctx.get_option("perm_mode")
    ctx.set_option("perm_mode", 2)
    try:
        with pytest.raises(capi.BisError):
            host.solve_block(ctx, "none", crs=(rp, col, val), B=B, method="gm")
    finally:
        ctx.set_option("perm_mode", old)


# ---- block GMRES against a per-column composition -----------------------------------------------------------
def composition(ctx, A, n, b, x0, precond, m, max_iters, tol):
    """GMRES on one column through the single-vector entry points, with the host's Givens update and the
    harness's stop and restart rules (host/methods/gmres.hpp, host/solver_harness.hpp)."""
    bb, x, x_old, tmp, r, w = ctx.upload(b), ctx.upload(x0), ctx.upload(x0), ctx.alloc(n), ctx.alloc(n), ctx.alloc(n)
    V = [ctx.alloc(n) for _ in range(m + 1)]   # every basis vector 16-byte aligned
    Vc = ctx.alloc((m + 1) * n)                # the contiguous basis bis_gmres_update_x reads
    D = None
    if precond == "j":
        D = ctx.alloc(n)
        ctx.call("bis_matrix_extract_diagonal", A.h, D, None)
    st = {}

    def reset():
        st.update(y=np.zeros(m + 1), H=np.zeros((m + 1) * m), H_tmp=np.zeros((m + 1) * m), R=np.zeros((m + 1) * m),
                  J=np.eye(m + 1).ravel().copy(), Q=np.eye(m + 1).ravel().copy(), Q_tmp=np.eye(m + 1).ravel().copy(),
                  g=np.zeros(m + 1), g_tmp=np.zeros(m + 1))

    def init_residual(first):
        ctx.call("bis_spmv", A.h, x, tmp)
        ctx.call("bis_subtract_vectors", r, bb, tmp, n, 1.0)
        ctx.call("bis_sumsq_to_slot", r, n, S_RR)
        if first:
            st["rn"] = math.sqrt(ctx.scalars(S_RR)[0])
            hist.append(st["rn"])
        if D:
            ctx.call("bis_elemwise_div_vectors", r, r, D, n, 1.0)
        ctx.call("bis_sumsq_to_slot", r, n, S_BETA2)
        ctx.call("bis_scale_inv_norm", n, V[0], r, S_BETA2)
        reset()
        st["beta"] = math.sqrt(ctx.scalars(S_BETA2)[0])
        st["g"][0] = st["g_tmp"][0] = st["beta"]
        if not first:
            st["rn"] = st["beta"]
            hist.append(st["beta"])

    def explicit_x(kk):
        host.gmres_back_substitution(kk, m, st["R"], st["g"], st["y"])
        for l in range(kk):
            ctx.call("bis_copy_vector", Vc + 8 * l * n, V[l], n)
        ctx.call("bis_gmres_update_x", n, kk, Vc, ptr(st["y"]), x, x_old, None)

    hist, it, restarts = [], 0, 0
    init_residual(True)
    thresh = tol * hist[0]
    while True:
        i = it - restarts * m
        ctx.call("bis_spmv", A.h, V[i], w)
        if D:
            ctx.call("bis_elemwise_div_vectors", w, w, D, n, 1.0)
        ctx.call("bis_dot_to_slot", w, V[0], n, S_H)
        for l in range(i + 1):
            ctx.call("bis_mgs_step", n, w, V[l], V[l + 1] if l < i else None, S_H + l, S_H + l + 1)
        ctx.call("bis_scale_inv_norm", n, V[i + 1], w, S_H + i + 1)
        col = ctx.scalars(S_H, i + 2)
        for l in range(i + 1):
            st["H"][i + l * m] = col[l]
        with np.errstate(invalid="ignore"):
            st["H"][(i + 1) * m + i] = np.sqrt(col[i + 1])
        host.gmres_least_squares(i, m, st["J"], st["H"], st["H_tmp"], st["Q"], st["Q_tmp"], st["R"])
        st["rn"] = host.gmres_update_g(i, m, st["Q"], st["g"], st["g_tmp"], st["beta"])
        it += 1
        hist.append(st["rn"])
        rn = st["rn"]
        if not (rn < thresh) and not (it > max_iters) and it % m == 0:   # check_restart
            explicit_x(it - restarts * m)
            ctx.call("bis_copy_vector", x_old, x, n)
            init_residual(False)
            restarts += 1
        rn = st["rn"]
        if abs(rn) < thresh or it >= max_iters - restarts or abs(rn) > np.finfo(float).max or math.isnan(rn):
            break
    explicit_x(it - restarts * m)   # save_x_star
    xs = ctx.download(x, n)
    for p in [bb, x, x_old, tmp, r, w, Vc] + V + ([D] if D else []):
        ctx.free(p)
    return np.array(hist), it, restarts, bool(rn < thresh), xs


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


def cap_for(mat, m):
    return {"random300": 60, "anderson_12_10_8": 60}.get(mat, 100 if m == 1 else 0)


def check_vs_composition(ctx, got, rp, col, val, B, X0, precond, m, max_iters, tol):
    n = len(rp) - 1
    A = ctx.upload_crs(rp, col, val)
    for j in range(B.shape[1]):
        hist, it, rst, conv, x = composition(ctx, A, n, B[:, j].copy(), X0[:, j].copy(), precond, m,
                                             max_iters or host.MAX_ITERS, tol)
        assert same(got.histories[j], hist), j
        assert (got.iter_counts[j], got.restarts[j], got.converged[j]) == (it, rst, conv), (j, it, rst, conv)
        assert same(got.x_star[:, j], x), j
    A.free()


@pytest.mark.parametrize("m", [1, 4, 10])
@pytest.mark.parametrize("precond", ["none", "j"])
@pytest.mark.parametrize("mat", ["hpcg32", "anderson_12_10_8", "random300"])
def test_block_gmres_vs_composition_bitwise(ctx, mat, precond, m):
    rp, col, val = named(mat)
    B, X0 = block_case(len(rp) - 1)
    tol, cap = 1e-8, cap_for(mat, m)
    got = host.solve_block(ctx, precond, crs=(rp, col, val), B=B, X0=X0, tol=tol, max_iters=cap, method="gm",
                           restart_len=m)
    check_vs_composition(ctx, got, rp, col, val, B, X0, precond, m, cap, tol)
    # the zero column stops on its NaN at iteration 1 without disturbing the others
    assert got.iter_counts[5] == 1 and np.isnan(got.histories[5][1]) and not got.converged[5]
    assert all(np.all(np.isfinite(got.histories[j])) for j in range(8) if j != 5)
    if mat == "hpcg32" and m > 1:
        # the columns converge in different restart cycles, some of them in the middle of a cycle
        assert all(got.converged[j] for j in range(8) if j != 5)
        assert len(set(int(v) for v in got.restarts)) >= 3, got.restarts
        assert any(int(v) % m for v in got.iter_counts if v > 1), got.iter_counts


# ---- against the single-RHS solve and the oracle --------------------------------------------------------------
ANDERSON = "Anderson,Lx=16,Ly=12,Lz=10,ranpot=5.0,t=1.0,seed=1"


@pytest.mark.parametrize("mat,precond", [("hpcg32", "none"), ("hpcg32", "j"), (ANDERSON, "j")])
def test_block_gmres_vs_single_rhs_and_oracle(ctx, mat, precond):
    m, k, tol = 10, 4, 1e-10
    if mat == "hpcg32":
        rp, col, val = named(mat)
        kw, max_iters = dict(crs=(rp, col, val)), 0
    else:
        rp, col, val = host.matrix(mat)
        kw, max_iters = dict(matrix_name=mat), 150
    n = len(rp) - 1
    B = np.random.default_rng(5).uniform(-1, 1, (n, k))
    B[:, 0] = 1.0
    X0 = np.full((n, k), 0.1)
    X0[:, -1] = np.random.default_rng(6).uniform(0, 1, n)
    got = host.solve_block(ctx, precond, B=B, X0=X0, tol=tol, max_iters=max_iters, method="gm", restart_len=m, **kw)
    for j in range(k):
        ref = port.solve(rp, col, val, "gm", precond, restart_len=m, b=B[:, j], x0=X0[:, j], tol=tol,
                         max_iters=max_iters)
        one = host.solve(ctx, "gm", precond, restart_len=m, b=B[:, j], x0=X0[:, j], tol=tol, max_iters=max_iters, **kw)
        r0 = ref.history[0]
        for other in (ref, one):
            assert (got.iter_counts[j], got.restarts[j]) == (other.iter_count, other.restarts), (j, other.iter_count)
            assert got.histories[j].size == other.history.size
            assert np.max(np.abs(got.histories[j] - other.history)) <= 1e-10 * r0, j
            assert got.converged[j] == other.converged
        if ref.converged:
            assert np.max(np.abs(got.x_star[:, j] - ref.x_star)) <= 1e-9 * max(np.max(np.abs(ref.x_star)), 1.0), j
        assert abs(got.final_true_residuals[j] - ref.final_true_residual) <= 1e-10 * r0, j


# ---- invariance -----------------------------------------------------------------------------------------------
def test_block_gmres_invariance_bitwise(ctx):
    rp, col, val = named("hpcg32")
    n = len(rp) - 1
    B, X0 = block_case(n)
    crs = (rp, col, val)
    kw = dict(crs=crs, tol=1e-8, method="gm", restart_len=10)
    base = host.solve_block(ctx, "j", B=B, X0=X0, **kw)

    def eq(r, j, s, i):
        return (same(r.histories[j], s.histories[i]) and r.iter_counts[j] == s.iter_counts[i]
                and r.restarts[j] == s.restarts[i] and r.converged[j] == s.converged[i]
                and same(r.x_star[:, j], s.x_star[:, i]))

    perm = np.array([3, 7, 0, 5, 1, 6, 2, 4])
    pr = host.solve_block(ctx, "j", B=B[:, perm], X0=X0[:, perm], **kw)
    assert all(eq(pr, i, base, perm[i]) for i in range(8))
    for j in (0, 2, 5):
        one = host.solve_block(ctx, "j", B=B[:, j:j + 1], X0=X0[:, j:j + 1], **kw)
        assert eq(one, 0, base, j), j
    old = ctx.get_option("graph")
    try:
        ctx.set_option("graph", 1 - old)
        other = host.solve_block(ctx, "j", B=B, X0=X0, **kw)
    finally:
        ctx.set_option("graph", old)
    again = host.solve_block(ctx, "j", B=B, X0=X0, **kw)
    assert all(eq(other, j, base, j) and eq(again, j, base, j) for j in range(8))
    # a max_iters cap that lands in the middle of a restart cycle
    cap = host.solve_block(ctx, "j", B=B, X0=X0, crs=crs, tol=1e-8, method="gm", restart_len=10, max_iters=37)
    assert all(int(v) % 10 for v in cap.iter_counts if v > 1), cap.iter_counts
    check_vs_composition(ctx, cap, rp, col, val, B, X0, "j", 10, 37, 1e-8)


# ---- shape ------------------------------------------------------------------------------------------------------
def test_block_gmres_launches_profile_and_memory(ctx, no_vector_cache):
    rp, col, val = named("hpcg32")
    n = len(rp) - 1
    crs = (rp, col, val)
    B, X0 = np.ones((n, 3)), np.full((n, 3), 0.1)
    kw = dict(crs=crs, B=B, X0=X0, tol=1e-30, method="gm", restart_len=10, max_iters=7)
    got = host.solve_block(ctx, "none", **kw)
    assert list(got.iter_counts) == [7, 7, 7] and list(got.restarts) == [0, 0, 0] and got.iterations == 7
    # set-up 4 (SpMM, residual, beta, V_0), basis index i: i + 4, the final x: 1
    assert got.launches == 4 + sum(i + 4 for i in range(7)) + 1, got.launches
    ctx.profile_enable(True)
    try:
        host.solve_block(ctx, "none", **kw)
        _, cnt = ctx.profile_read("spmv")
    finally:
        ctx.profile_enable(False)
    assert cnt == 1 + 7 + 1   # set-up, one per iteration, the true residual
    # device memory comes back: a second solve of the same shape (graphs recorded, Jacobi diagonal) ends where
    # the first left it
    host.solve_block(ctx, "j", **dict(kw, max_iters=25))
    ctx.sync()
    free0 = ctx.info()["free"]
    host.solve_block(ctx, "j", **dict(kw, max_iters=25))
    ctx.sync()
    assert ctx.info()["free"] == free0
    # without `method`, solve_block is the block CG
    cg = host.solve_block(ctx, "none", crs=crs, B=B, X0=X0, max_iters=5, tol=1e-30)
    assert cg.restarts is None and list(cg.iter_counts) == [5, 5, 5]
