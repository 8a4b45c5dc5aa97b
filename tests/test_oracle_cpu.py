"""CPU tests that PIN THE ORACLE (oracle/port, the plain-C restatement):
 (1) against the reference's own known-answer tests (tests/test_kernels.cpp,
     tests/test_utilities.cpp, tests/test_solvers.cpp under /root/reference), restated here;
 (2) against fixtures produced by the compiled, unmodified reference
     (tests/golden/*.npz, made by tests/golden/make_golden.py);
 (3) live against oracle/_ref/libbis_ref.so when it is present (build container).
Bit-exact where the summation order is defined (triangular solves, axpby family, ILU(0));
1e-10 * ||r0|| for residual histories (north_star's tolerance); 1e-13 relative for
SpMV/dot/norm whose order the reference leaves to OpenMP/SIMD (SURVEY.md F12).
"""
import numpy as np
import pytest

from conftest import HIST_TOL, check_against_fixture, golden
from oracle import matgen, port, refshim

RED_TOL = 1e-13    # relative, order-unspecified reductions


def i32(*a):
    return np.array(a, np.int32)


def f64(*a):
    return np.array(a, np.float64)


# ---- (1) reference known-answer tests -------------------------------------------------
def test_kat_spmv_diag_and_dense():
    # tests/test_kernels.cpp:26-66
    y = port.spmv(i32(0, 1, 2, 3), i32(0, 1, 2), f64(2, 3, 4), f64(1, 2, 3))
    assert np.array_equal(y, f64(2, 6, 12))
    y = port.spmv(i32(0, 3, 6, 9), i32(0, 1, 2, 0, 1, 2, 0, 1, 2), f64(*range(1, 10)), f64(1, 2, 3))
    assert np.array_equal(y, f64(14, 32, 50))


def test_kat_sptrsv_forward_backward():
    # tests/test_kernels.cpp:69-93 and :96-120
    x = port.sptrsv(i32(0, 0, 1, 3), i32(0, 0, 1), f64(1, -2, 1), f64(2, 3, 4), f64(2, 7, 12))
    assert np.allclose(x, f64(1, 2, 3), atol=1e-9)
    x = port.sptrsv(i32(0, 2, 3, 3), i32(1, 2, 2), f64(1, -2, 1), f64(2, 3, 4), f64(-2, 9, 12), backward=True)
    assert np.allclose(x, f64(1, 2, 3), atol=1e-9)


def test_kat_vector_ops():
    # tests/test_kernels.cpp:122-154
    lib = port.load()
    a, b = f64(1, 2, 3), f64(4, 5, 6)
    out = np.zeros(3)
    lib.o_sum_vectors(out, a, b, 3, 2.0)
    assert np.array_equal(out, f64(9, 12, 15))
    lib.o_subtract_vectors(out, a, b, 3, 2.0)
    assert np.array_equal(out, f64(-7, -8, -9))
    lib.o_elemwise_mult_vectors(out, a, b, 3, 1.0)
    assert np.array_equal(out, f64(4, 10, 18))
    lib.o_elemwise_div_vectors(out, b, a, 3, 1.0)
    assert np.allclose(out, f64(4, 2.5, 2), atol=1e-12)
    assert lib.o_dot(f64(1, 2, 3), f64(2, 4, 5), 3) == 25.0
    lib.o_scale(out, a, 3.0, 3)
    assert np.array_equal(out, f64(3, 6, 9))


def test_kat_norm_including_empty():
    # tests/test_utilities.cpp:34-62
    lib = port.load()
    assert lib.o_euclidean_vec_norm(f64(3, 4), 2) == 5.0
    assert lib.o_euclidean_vec_norm(f64(0.0), 0) == 0.0


def _dense3():
    rp = i32(0, 3, 6, 9)
    col = i32(0, 1, 2, 0, 1, 2, 0, 1, 2)
    val = f64(1, 2, 3, 4, 5, 6, 7, 8, 9)
    return rp, col, val


def test_kat_split_and_peel():
    # tests/test_utilities.cpp:96-208: strict parts and the diagonal of a dense 3x3
    f = port.factor(*_dense3(), "none")
    assert np.array_equal(f.l_rp, i32(0, 0, 1, 3)) and np.array_equal(f.l_col, i32(0, 0, 1))
    assert np.array_equal(f.l_val, f64(4, 7, 8))
    assert np.array_equal(f.u_rp, i32(0, 2, 3, 3)) and np.array_equal(f.u_col, i32(1, 2, 2))
    assert np.array_equal(f.u_val, f64(2, 3, 6))
    assert np.array_equal(f.A_D, f64(1, 5, 9))
    assert np.allclose(f.A_D_inv, 1.0 / f64(1, 5, 9), rtol=0, atol=0)


def test_kat_preconditioner_none_jacobi_gs_bgs():
    # tests/test_kernels.cpp:156-225
    rp, col, val = i32(0, 1, 3, 6), i32(0, 0, 1, 0, 1, 2), f64(2, 1, 3, -2, 1, 4)   # lower-triangular A
    f = port.factor(rp, col, val, "gs")
    v = f64(2, 7, 12)
    assert np.array_equal(port.apply_preconditioner("none", f, v), v)
    assert np.allclose(port.apply_preconditioner("j", f, v), v / f64(2, 3, 4), atol=1e-12)
    assert np.allclose(port.apply_preconditioner("gs", f, v), f64(1, 2, 3), atol=1e-9)
    rp, col, val = i32(0, 3, 5, 6), i32(0, 1, 2, 1, 2, 2), f64(2, 1, -2, 3, 1, 4)   # upper-triangular A
    f = port.factor(rp, col, val, "bgs")
    assert np.allclose(port.apply_preconditioner("bgs", f, f64(-2, 9, 12)), f64(1, 2, 3), atol=1e-9)


@pytest.mark.parametrize("method,pre", [("cg", "none"), ("cg", "j"), ("bi", "none"), ("bi", "j"),
                                        ("j", "none"), ("gs", "none"), ("sgs", "none")])
def test_kat_3x3_solves(method, pre):
    # tests/test_solvers.cpp:49-91,158-192: tridiag(-1,2,-1), x_true=[1,2,3], b=[0,0,4], x0=0
    rp, col, val = i32(0, 2, 5, 7), i32(0, 1, 0, 1, 2, 1, 2), f64(2, -1, -1, 2, -1, -1, 2)
    r = port.solve(rp, col, val, method, pre, b=f64(0, 0, 4), x0=f64(0, 0, 0))
    assert r.converged
    assert np.max(np.abs(r.x_star - f64(1, 2, 3))) <= 1e-7


def test_kat_3x3_bicgstab_jacobi_diag10():
    # tests/test_solvers.cpp:93-141: tridiag(-1,10,-1)
    rp, col, val = i32(0, 2, 5, 7), i32(0, 1, 0, 1, 2, 1, 2), f64(10, -1, -1, 10, -1, -1, 10)
    xt = f64(1, 2, 3)
    b = port.spmv(rp, col, val, xt)
    r = port.solve(rp, col, val, "bi", "j", b=b, x0=f64(0, 0, 0))
    assert r.converged and np.max(np.abs(r.x_star - xt)) <= 1e-7


# ---- (2) fixtures produced by the compiled reference ----------------------------------------
def _matrix(name, g):
    if name == "hpcg16":
        return matgen.hpcg(16)
    if name == "hpcg32":
        return matgen.hpcg(32)
    return g["rp"], g["col"], g["val"]


@pytest.mark.parametrize("name", ["fdm2d16", "band_klein", "hpcg16"])
def test_golden_kernels(name):
    g = golden(name)
    rp, col, val = _matrix(name, g)
    x, v = g["k__x"], g["k__v"]
    n = x.size
    lib = port.load()
    assert np.array_equal(port.spmv(rp, col, val, x), g["k__spmv"])
    f = port.factor(rp, col, val, "sgs")
    if "k__split__l_rp" in g:
        for k in ("l_rp", "l_col", "l_val", "u_rp", "u_col", "u_val", "A_D", "A_D_inv"):
            assert np.array_equal(getattr(f, k), g["k__split__" + k]), k
    # triangular solves and every preconditioner built from them: bit-exact
    assert np.array_equal(port.sptrsv(f.l_rp, f.l_col, f.l_val, f.A_D, x), g["k__sptrsv"])
    assert np.array_equal(port.sptrsv(f.u_rp, f.u_col, f.u_val, f.A_D, x, backward=True), g["k__bsptrsv"])
    assert np.array_equal(port.sptrsv_inplace(f.l_rp, f.l_col, f.l_val, f.A_D, x), g["k__sptrsv_inplace"])
    for pre in ("none", "j", "gs", "bgs", "sgs"):
        assert np.array_equal(port.apply_preconditioner(pre, f, x), g["k__precond__" + pre]), pre
    fi = port.factor(rp, col, val, "ilu0")
    assert np.array_equal(fi.L_D, g["k__ilu0__L_D"])
    assert np.array_equal(fi.U_D, g["k__ilu0__U_D"])
    assert np.array_equal(fi.u_val, g["k__ilu0__u_val"])
    if "k__ilu0__l_val" in g:
        assert np.array_equal(fi.l_val, g["k__ilu0__l_val"])
    assert np.array_equal(port.apply_preconditioner("ilu0", fi, x), g["k__precond__ilu0"])
    # axpby family: bit-exact
    for fn in ("subtract_vectors", "sum_vectors", "elemwise_mult_vectors", "elemwise_div_vectors"):
        o = np.zeros(n)
        getattr(lib, "o_" + fn)(o, x, v + 2.0, n, 0.37)
        assert np.array_equal(o, g["k__" + fn]), fn
    o = np.zeros(n)
    lib.o_scale(o, x, -1.25, n)
    assert np.array_equal(o, g["k__scale"])
    assert abs(lib.o_dot(x, v, n) - g["k__dot"][0]) <= RED_TOL * np.sqrt(n)
    assert abs(lib.o_euclidean_vec_norm(x, n) - g["k__norm"][0]) <= RED_TOL * g["k__norm"][0]
    xn = port.spmv(rp, col, val, x)
    lib.o_normalize_x(xn, x, f.A_D, v, n)
    assert np.array_equal(xn, g["k__normalize_x"])


def _solve_keys(g):
    return sorted(k[:-len("__history")] for k in g.files if k.endswith("__history"))


@pytest.mark.parametrize("name", ["fdm2d16", "band_klein", "hpcg16", "hpcg32", "anderson_12_10_8",
                                  "anderson_dd_12_10_8"])
def test_golden_solves(name):
    g = golden(name)
    rp, col, val = _matrix(name, g)
    for key in _solve_keys(g):
        method, pre = key.split("__")
        if name == "hpcg16" and method in ("j", "gs", "sgs"):
            continue   # ~1000 serial sweeps each; covered by fdm2d16 / band_klein
        got = port.solve(rp, col, val, method, pre)
        check_against_fixture(got, g, key)


# ---- (3) a random sparsity pattern: stored fixture, and live against the compiled reference where it is built ----
def _dense(rp, col, val, n):
    d = np.zeros((n, n))
    d[np.repeat(np.arange(n), np.diff(rp)), col] = val
    return d


def test_live_reference_random_matrix():
    """Symmetric diagonally dominant 300 x 300 matrix with a random pattern (tests/golden/make_golden.py random300):
    the oracle against the stored ILU(0) factors, preconditioner outputs and solves (bit-exact / 1e-10 * ||r0||,
    same counts); the stored values against their defining equations in dense arithmetic; and, where oracle/_ref is
    built, the oracle against the compiled reference live."""
    g = golden("random300")
    rp, col, val, x = g["rp"], g["col"], g["val"], g["x"]
    n = rp.size - 1
    fp = port.factor(rp, col, val, "ilu0")
    for k in ("l_rp", "l_col", "l_val", "u_rp", "u_col", "u_val", "L_D", "U_D"):
        assert np.array_equal(getattr(fp, k), g["ilu0__" + k]), k
    assert np.array_equal(port.apply_preconditioner("ilu0", fp, x), g["precond__ilu0"])
    assert np.array_equal(port.apply_preconditioner("sgs", port.factor(rp, col, val, "sgs"), x), g["precond__sgs"])
    for key in sorted(k[:-len("__history")] for k in g.files if k.endswith("__history")):
        method, pre = key.split("__")
        r, want = port.solve(rp, col, val, method, pre), g[key + "__history"]
        its, conv, restarts = (int(v) for v in g[key + "__meta"])
        assert (r.iter_count, r.converged, r.restarts) == (its, bool(conv), restarts), key
        assert r.history.size == want.size and np.max(np.abs(r.history - want)) <= HIST_TOL * want[0], key

    # the stored values in dense arithmetic: ILU(0) reproduces A on its pattern, the preconditioner outputs solve
    # their systems, every history starts at ||b - A x0|| (b = 1, x0 = 0.1) and the solves converged
    A = _dense(rp, col, val, n)
    L = np.eye(n) + _dense(g["ilu0__l_rp"], g["ilu0__l_col"], g["ilu0__l_val"], n)
    U = np.diag(g["ilu0__U_D"]) + _dense(g["ilu0__u_rp"], g["ilu0__u_col"], g["ilu0__u_val"], n)
    assert np.array_equal(g["ilu0__L_D"], np.ones(n))
    assert np.max(np.abs((L @ U - A)[A != 0])) <= 1e-13 * np.max(np.abs(A))
    assert np.linalg.norm(L @ U @ g["precond__ilu0"] - x) <= 1e-13 * np.linalg.norm(x)
    M = np.tril(A) @ np.diag(1.0 / np.diag(A)) @ np.triu(A)             # (D + L) D^-1 (D + U)
    assert np.linalg.norm(M @ g["precond__sgs"] - x) <= 1e-13 * np.linalg.norm(x)
    r0 = np.linalg.norm(np.ones(n) - A @ np.full(n, 0.1))
    for key in (k[:-len("__history")] for k in g.files if k.endswith("__history")):
        h = g[key + "__history"]
        assert abs(h[0] - r0) <= 1e-13 * r0 and g[key + "__meta"][1] == 1 and h[-1] < 1e-14 * h[0], key

    if not refshim.available():
        return
    refshim.load().ref_omp_set_threads(1)
    fr = refshim.factor(rp, col, val, "ilu0")
    for k in ("l_val", "u_val", "L_D", "U_D"):
        assert np.array_equal(getattr(fr, k), getattr(fp, k)), k
    for pre in ("sgs", "ilu0"):
        f_r = fr if pre == "ilu0" else refshim.factor(rp, col, val, pre)
        f_p = fp if pre == "ilu0" else port.factor(rp, col, val, pre)
        assert np.array_equal(refshim.apply_preconditioner(pre, f_r, x), port.apply_preconditioner(pre, f_p, x))
    for method, pre in (("cg", "sgs"), ("bi", "ilu0"), ("gm", "ilu0"), ("sgs", "none")):
        a = refshim.solve(rp, col, val, method, pre, threads=1)
        b = port.solve(rp, col, val, method, pre)
        assert a.iter_count == b.iter_count
        assert np.max(np.abs(a.history - b.history)) <= HIST_TOL * a.history[0]


@pytest.mark.parametrize("name", ["fdm2d16_scale", "anderson_dd_12_10_8_scale"])
def test_scale_restatement_against_reference_fixtures(name):
    """-scale 1: the numpy restatement of extract_scale/scale_mat (oracle/port.py) feeding the oracle
    reproduces the compiled reference's scaled solves (tests/golden/make_golden.py scale)."""
    g = golden(name)
    val_s, sc = port.scale_symmetric(g["rp"], g["col"], g["val"])
    n = len(g["rp"]) - 1
    for key in sorted(k[:-len("__history")] for k in g.files if k.endswith("__history")):
        method, pre = key.split("__")
        r = port.solve(g["rp"], g["col"], val_s, method, pre, b=sc * np.ones(n), x0=np.full(n, 0.1))
        want = g[key + "__history"]
        k = min(want.size, r.history.size)
        assert np.max(np.abs(r.history[:k] - want[:k])) <= 1e-10 * want[0], key
        assert r.iter_count == int(g[key + "__meta"][0]), key
