"""Grid tiles of the windowed SpMV (csrc/bis_spmv_win.cuh, WinFormat::grid): a matrix on its generator's grid hint
with R | nx, every nonzero in its row's 27-point stencil, ascending columns and at most 256 row patterns streams a
class byte per row and fetches x as one 3-D box per tile.  The format is chosen from the matrix alone; every fused
form must keep the oracle's bits, and the fused dot products must keep the bits of the window format, because the
tile, CTA, group and thread mapping is the same."""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import matgen, port

pytestmark = pytest.mark.gpu

WINDOWS, GRID = 3, 4


@pytest.fixture(autouse=True)
def _options(ctx):
    saved = {k: ctx.get_option(k) for k in ("spmv_variant", "spmv_vdict")}
    ctx.set_option("spmv_variant", 3)
    yield
    for k, v in saved.items():
        ctx.set_option(k, v)


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def crs32(A):
    rp, col, val = A.download()
    return rp.astype(np.int32), col, val


def fused_forms(ctx, A, x, v, D):
    """y of bis_spmv and of every fused form, the reduced scalars, and the format / byte model of the bis_spmv launch"""
    n = x.size
    dx, dv, dD = ctx.upload(x), ctx.upload(v), ctx.upload(D)
    dy, dr, dt, dxn = (ctx.alloc(n) for _ in range(4))
    out = {}
    try:
        ctx.call("bis_spmv", A.h, dx, dy)
        out["spmv"] = ctx.download(dy, n)
        out["format"], out["mb"] = ctx.get_option("spmv_format"), ctx.get_option("spmv_stream_mb")
        out["value_bytes"] = ctx.get_option("spmv_value_bytes")
        ctx.call("bis_spmv_dot", A.h, dx, dy, dv, 20, 21)
        out["dot_y"], out["dot_s"] = ctx.download(dy, n), ctx.scalars(20, 2)
        ctx.call("bis_spmv_dot", A.h, dx, dy, dx, 22, 23)
        out["dotx_y"], out["dotx_s"] = ctx.download(dy, n), ctx.scalars(22, 2)
        ctx.call("bis_spmv_residual", A.h, dx, dv, dr, dt, 24)
        out["res_r"], out["res_t"], out["res_s"] = ctx.download(dr, n), ctx.download(dt, n), ctx.scalars(24)
        ctx.call("bis_spmv_jacobi", A.h, dD, dv, dx, dxn)
        out["jac"] = ctx.download(dxn, n)
        ctx.call("bis_spmv_jacobi_residual", A.h, dD, dv, dx, dxn, dr, 25)
        out["jacr_x"], out["jacr_r"], out["jacr_s"] = ctx.download(dxn, n), ctx.download(dr, n), ctx.scalars(25)
    finally:
        for d in (dx, dv, dD, dy, dr, dt, dxn):
            ctx.free(d)
    return out


def check_against_oracle(out, rp, col, val, x, v, D):
    y = port.spmv(rp, col, val, x)
    for k in ("spmv", "dot_y", "dotx_y", "res_t"):
        assert np.array_equal(bits(out[k]), bits(y)), k
    for k in ("res_r", "jacr_r"):
        assert np.array_equal(bits(out[k]), bits(v - y)), k
    jac = (v - (y - D * x)) / D
    for k in ("jac", "jacr_x"):
        assert np.array_equal(bits(out[k]), bits(jac)), k
    assert abs(out["dot_s"][0] - y @ v) <= 1e-12 * np.linalg.norm(y) * np.linalg.norm(v)
    assert abs(out["dotx_s"][0] - y @ x) <= 1e-12 * np.linalg.norm(y) * np.linalg.norm(x)


def vectors(n, seed=5):
    rng = np.random.default_rng(seed)
    return rng.uniform(-1.0, 1.0, n), rng.uniform(-1.0, 1.0, n), rng.uniform(1.0, 2.0, n)


def stream_mb(value_bytes, rp_bytes, n, nnz, grid):
    """the byte model of bis_spmv (EpiStore: y) in units of 1e6 bytes"""
    b = value_bytes * nnz + (n if grid else 2 * nnz) + rp_bytes * (n + 1) + 8 * (n + n)
    return (b + 500000) // 1000000


GRID_CASES = {
    "hpcg_128": lambda ctx: ctx.generate_hpcg(128, 128, 128),
    "hpcg_256_8_6": lambda ctx: ctx.generate_hpcg(256, 8, 6),
    "hpcg_384_5_130": lambda ctx: ctx.generate_hpcg(384, 5, 130),
    "anderson_256_6_5": lambda ctx: ctx.generate_anderson(256, 6, 5, 5.0, 1.0, 3, False),
}


@pytest.mark.parametrize("name", sorted(GRID_CASES))
def test_grid_tiles_are_taken_and_keep_the_bits(ctx, name):
    A = GRID_CASES[name](ctx)
    try:
        rp, col, val = crs32(A)
        rp_bytes = A.info()["rp_bytes"]
        n = rp.size - 1
        x, v, D = vectors(n)
        runs = {}
        for vdict in (1, 0):
            ctx.set_option("spmv_vdict", vdict)
            runs[vdict] = fused_forms(ctx, A, x, v, D)
    finally:
        A.free()
    dict_bytes = 8 if name.startswith("anderson") else 1      # the Anderson diagonal has more than 256 values
    for vdict, vb in ((1, dict_bytes), (0, 8)):
        out = runs[vdict]
        assert out["format"] == GRID, (vdict, out["format"])
        assert out["value_bytes"] == vb
        assert out["mb"] == stream_mb(vb, rp_bytes, n, col.size, True)
        check_against_oracle(out, rp, col, val, x, v, D)
    for k in runs[0]:
        if k not in ("value_bytes", "mb"):
            assert np.array_equal(np.asarray(runs[1][k]).view(np.uint64), np.asarray(runs[0][k]).view(np.uint64)), k


def _permuted_hpcg():
    rp, col, val = matgen.hpcg(128, 4, 3)
    n = rp.size - 1
    perm = np.random.default_rng(2).permutation(n)
    P = sp.csr_matrix((val, col, rp), shape=(n, n))[perm][:, perm].tocsr()
    P.sort_indices()
    return P.indptr.astype(np.int32), P.indices.astype(np.int32), P.data


WINDOW_CASES = {
    "generated_hpcg_130_7_5": lambda ctx: ctx.generate_hpcg(130, 7, 5),           # R does not divide nx
    "uploaded_hpcg_128_4_3": lambda ctx: ctx.upload_crs(*matgen.hpcg(128, 4, 3)),  # no grid hint
    "uploaded_permuted_hpcg": lambda ctx: ctx.upload_crs(*_permuted_hpcg()),
}


@pytest.mark.parametrize("name", sorted(WINDOW_CASES))
def test_other_matrices_keep_windows(ctx, name):
    A = WINDOW_CASES[name](ctx)
    try:
        rp, col, val = crs32(A)
        rp_bytes = A.info()["rp_bytes"]
        x, v, D = vectors(rp.size - 1)
        ctx.set_option("spmv_vdict", 1)
        out = fused_forms(ctx, A, x, v, D)
    finally:
        A.free()
    assert out["format"] == WINDOWS
    assert out["mb"] == stream_mb(1, rp_bytes, rp.size - 1, col.size, False)
    check_against_oracle(out, rp, col, val, x, v, D)


def test_split_factor_takes_grid_tiles(ctx):
    """the strict triangles of a generated grid matrix carry its hint: b - U x runs on grid tiles"""
    A = ctx.generate_hpcg(128, 6, 5)
    L, U = ctx.split_triangular(A)
    try:
        rp, col, val = crs32(U)
        n = rp.size - 1
        x, v, _ = vectors(n)
        dx, dv, dout = ctx.upload(x), ctx.upload(v), ctx.alloc(n)
        ctx.call("bis_spmv_sub", U.h, dx, dv, dout)
        got, fmt = ctx.download(dout, n), ctx.get_option("spmv_format")
        for d in (dx, dv, dout):
            ctx.free(d)
    finally:
        for M in (L, U, A):
            M.free()
    assert fmt == GRID
    assert np.array_equal(bits(got), bits(v - port.spmv(rp, col, val, x)))


@pytest.mark.parametrize("nx", [128, 256])
def test_reduced_scalars_equal_those_of_windows(ctx, nx):
    """HPCG-128 and HPCG-256 have one traversal block, so the order table is natural with and without the grid
    hint: the generated matrix (grid tiles) and the same CRS uploaded (windows) reduce the same per-thread sums"""
    G = ctx.generate_hpcg(nx, nx, nx)
    rp, col, val = crs32(G)
    W = ctx.upload_crs(rp, col, val)
    del col, val
    n = rp.size - 1
    x, v, D = vectors(n, seed=9)
    dx, dv, dD = ctx.upload(x), ctx.upload(v), ctx.upload(D)
    dy, dr, dxn = ctx.alloc(n), ctx.alloc(n), ctx.alloc(n)
    try:
        for vdict in (1, 0):
            ctx.set_option("spmv_vdict", vdict)
            s, fmt = {}, {}
            for tag, M in (("grid", G), ("win", W)):
                ctx.call("bis_spmv_dot", M.h, dx, dy, dv, 20, 21)
                fmt[tag] = ctx.get_option("spmv_format")
                ctx.call("bis_spmv_dot", M.h, dx, dy, dx, 22, 23)
                ctx.call("bis_spmv_residual", M.h, dx, dv, dr, 0, 24)
                ctx.call("bis_spmv_jacobi_residual", M.h, dD, dv, dx, dxn, dr, 25)
                s[tag] = ctx.scalars(20, 6)
            assert fmt == {"grid": GRID, "win": WINDOWS}
            assert np.array_equal(bits(s["grid"]), bits(s["win"])), (vdict, s)
    finally:
        for d in (dx, dv, dD, dy, dr, dxn):
            ctx.free(d)
        G.free()
        W.free()


def _release_vector_cache(ctx):
    on = ctx.get_option("vector_cache")
    ctx.set_option("vector_cache", 0)
    ctx.set_option("vector_cache", on)


def test_freeing_a_grid_matrix_returns_its_row_classes(ctx):
    """the class bytes (one per row, 16.8 MB here) go with the matrix"""
    def generate_use_free(nz):
        A = ctx.generate_hpcg(512, 512, nz)
        n = A.info()["n_rows"]
        dx, dy = ctx.alloc(n), ctx.alloc(n)
        ctx.call("bis_init_vector", dx, 1.0, n)
        ctx.call("bis_spmv", A.h, dx, dy)
        fmt = ctx.get_option("spmv_format")
        ctx.free(dx)
        ctx.free(dy)
        A.free()
        _release_vector_cache(ctx)
        return fmt

    generate_use_free(2)                  # first use: whatever the context sets up once
    free0 = ctx.info()["free"]
    assert generate_use_free(64) == GRID
    free1 = ctx.info()["free"]
    assert free1 >= free0 - (4 << 20), f"{(free0 - free1) / 2**20:.1f} MB stayed allocated"
