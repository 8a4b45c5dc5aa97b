"""The value dictionary is the windowed SpMV's default (csrc/bis_spmv.cu: win_build_dict).  Every fused form -- y, the
fused dot products (with w != x and with w == x, as CG calls it), residual and norm, the Jacobi forms, b - T x and the
two-stage form -- must have the bits of the value-streaming run and of the oracle, on HPCG grids, the Anderson matrix,
a banded matrix with more than 256 distinct values (no dictionary), empty rows, odd sizes and 32- / 64-bit row_ptr; and
whole solves must give identical histories and iterates with the dictionary on and off."""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import matgen, port

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _options(ctx):
    """the session's values of the options these tests set are restored afterwards (the suite may run with either
    dictionary setting, e.g. BIS_SPMV_VDICT=0)"""
    saved = {k: ctx.get_option(k) for k in ("spmv_variant", "spmv_vdict")}
    ctx.set_option("spmv_variant", 3)
    yield
    for k, v in saved.items():
        ctx.set_option(k, v)


def _banded_with_empty_rows(n, seed):
    """pentadiagonal, more than 256 distinct values, every 9th row empty"""
    rng = np.random.default_rng(seed)
    rows = [[] if r % 9 == 4 else [c for c in (r - 7, r - 1, r, r + 1, r + 7) if 0 <= c < n] for r in range(n)]
    rp = np.zeros(n + 1, np.int32)
    np.cumsum([len(c) for c in rows], out=rp[1:])
    col = np.array([c for cs in rows for c in cs], np.int32)
    val = rng.uniform(-2.0, 2.0, col.size)
    return rp, col, val


MATRICES = {
    "hpcg_20_14_11": lambda: matgen.hpcg(20, 14, 11),
    "hpcg_7_5_3_odd": lambda: matgen.hpcg(7, 5, 3),
    "hpcg_130_7_5": lambda: matgen.hpcg(130, 7, 5),
    "anderson": lambda: matgen.anderson(12, 10, 9, 5.0, 1.0, 7, False),
    "banded_empty_rows_odd": lambda: _banded_with_empty_rows(3001, 4),
}


def _fused_forms(ctx, A, T, x, v, D):
    """every fused form once; returns the outputs and the scalars they produced"""
    n = x.size
    dx, dv, dD = ctx.upload(x), ctx.upload(v), ctx.upload(D)
    dy, dr, dt, dxn, dout = (ctx.alloc(n) for _ in range(5))
    out = {}
    ctx.call("bis_spmv", A.h, dx, dy)
    out["spmv"] = ctx.download(dy, n)
    ctx.call("bis_spmv_dot", A.h, dx, dy, dv, 20, 21)
    out["dot_y"], out["dot_s"] = ctx.download(dy, n), ctx.scalars(20, 2)
    ctx.call("bis_spmv_dot", A.h, dx, dy, dx, 22, 23)
    out["dotx_s"] = ctx.scalars(22, 2)
    ctx.call("bis_spmv_residual", A.h, dx, dv, dr, dt, 24)
    out["res_r"], out["res_t"], out["res_s"] = ctx.download(dr, n), ctx.download(dt, n), ctx.scalars(24)
    ctx.call("bis_spmv_jacobi", A.h, dD, dv, dx, dxn)
    out["jac"] = ctx.download(dxn, n)
    ctx.call("bis_spmv_jacobi_residual", A.h, dD, dv, dx, dxn, dr, 25)
    out["jacr_x"], out["jacr_r"], out["jacr_s"] = ctx.download(dxn, n), ctx.download(dr, n), ctx.scalars(25)
    ctx.call("bis_spmv_sub", T.h, dx, dv, dr)
    out["sub"] = ctx.download(dr, n)
    ctx.upload(v * 0.5, dout)
    ctx.call("bis_spmv_two_stage", T.h, dD, dx, dt, dout)
    out["ts_w"], out["ts_out"] = ctx.download(dt, n), ctx.download(dout, n)
    for d in (dx, dv, dD, dy, dr, dt, dxn, dout):
        ctx.free(d)
    return out


@pytest.mark.parametrize("rp64", [False, True])
@pytest.mark.parametrize("name", sorted(MATRICES))
def test_fused_forms_have_the_bits_of_the_value_streaming_run(ctx, name, rp64):
    rp, col, val = MATRICES[name]()
    n = rp.size - 1
    if rp64:
        rp = rp.astype(np.int64)
    rng = np.random.default_rng(11)
    x, v, D = rng.uniform(-1.0, 1.0, n), rng.uniform(-1.0, 1.0, n), rng.uniform(1.0, 2.0, n)
    U = sp.triu(sp.csr_matrix((val, col, rp.astype(np.int32)), shape=(n, n)), 1).tocsr()
    U.sort_indices()
    u_rp, u_col, u_val = U.indptr.astype(np.int32), U.indices.astype(np.int32), U.data
    runs, value_bytes = {}, {}
    for vdict in (1, 0):
        ctx.set_option("spmv_vdict", vdict)
        A = ctx.upload_crs(rp, col, val)
        T = ctx.upload_triangular(u_rp, u_col, u_val, upper=True)
        runs[vdict] = _fused_forms(ctx, A, T, x, v, D)
        value_bytes[vdict] = ctx.get_option("spmv_value_bytes")     # of the last launch: T x
        A.free()
        T.free()
    assert value_bytes[0] == 8
    assert value_bytes[1] == (8 if name == "banded_empty_rows_odd" else 1)
    y_ref = port.spmv(rp.astype(np.int32), col, val, x)
    ref = runs[0]
    assert np.array_equal(ref["spmv"], y_ref)
    assert np.array_equal(ref["dot_y"], y_ref)
    assert np.array_equal(ref["res_r"], v - y_ref) and np.array_equal(ref["res_t"], y_ref)
    assert np.array_equal(ref["jac"], ref["jacr_x"])
    assert np.array_equal(ref["jacr_r"], v - y_ref)
    assert np.array_equal(ref["sub"], v - port.spmv(u_rp, u_col, u_val, x))
    assert abs(ref["dot_s"][0] - y_ref @ v) <= 1e-12 * np.linalg.norm(y_ref) * np.linalg.norm(v)
    assert abs(ref["dotx_s"][0] - y_ref @ x) <= 1e-12 * np.linalg.norm(y_ref) * np.linalg.norm(x)
    for k in ref:
        assert np.array_equal(runs[1][k].view(np.uint64), ref[k].view(np.uint64)), k


def test_hpcg48_solves_bit_identical_with_and_without_dictionary(ctx):
    """Whole solves: fused dot / Jacobi / residual epilogues inside the graph-replayed loop."""
    from basic_iterative_solvers_b200 import host
    ctx.set_option("spmv_variant", 0)
    out = {}
    for vdict in (1, 0):
        ctx.set_option("spmv_vdict", vdict)
        out[vdict] = [host.solve(ctx, m, p, matrix_name="HPCG-48", tol=1e-12, want_x=True)
                      for m, p in (("cg", "j"), ("bi", "j"), ("j", "none"))]
    for a, b in zip(out[1], out[0]):
        assert np.array_equal(a.history, b.history)
        assert np.array_equal(a.x_star, b.x_star)
