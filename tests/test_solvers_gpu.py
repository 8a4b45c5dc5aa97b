"""GPU parity tests, solver level: whole solves through the C++ host stack
(host/solver_harness.hpp, host/methods/*.hpp) and the C-ABI, compared with

 - the fixtures produced by the compiled, unmodified reference (tests/golden/*.npz), and
 - the oracle (oracle/port) run here on the same seeded inputs.

The bar is north_star's: iteration counts identical and max_k |r_k - r_k^ref| <= 1e-10 * ||r0||
(fp64).  The reference's own tests only pin 3x3 solutions to 1e-7 (tests/test_solvers.cpp);
those are reproduced through the device path as well.
"""
import numpy as np
import pytest

from conftest import HIST_TOL, check_against_fixture, golden
from oracle import matgen, port

from basic_iterative_solvers_b200 import capi, host

pytestmark = pytest.mark.gpu

def i32(*a):
    return np.array(a, np.int32)


def f64(*a):
    return np.array(a, np.float64)


def crossings(h):
    """First index where ||r_k|| / ||r_0|| drops below 1e-3, 1e-6, 1e-9 (the harness's res3/res6
    milestones, solver_harness.hpp:27-37, plus one deeper)."""
    out = []
    for lvl in (1e-3, 1e-6, 1e-9):
        below = np.nonzero(h / h[0] < lvl)[0]
        out.append(int(below[0]) if below.size else -1)
    return out


def check(got, want, exact_count=True):
    """GPU vs oracle on the same inputs.  History within 1e-10 * ||r0|| over the common prefix and
    identical milestone crossings always.  The iteration count at the stopping threshold is compared
    exactly when the threshold sits above the rounding floor (tests pass tol >= 1e-10); at the
    shipped TOL = 1e-14 the reference's own count moves with its OpenMP thread count (SURVEY.md F7;
    HPCG-128 -cg: 275..290 over 1/2/4/8 threads), so there it is compared within 5 % (at least 2)."""
    r0 = want.history[0]
    k = min(got.history.size, want.history.size)
    err = np.max(np.abs(got.history[:k] - want.history[:k])) / r0
    assert err <= HIST_TOL, err
    assert crossings(got.history) == crossings(want.history)
    assert got.converged == want.converged
    if exact_count:
        assert got.iter_count == want.iter_count and got.restarts == want.restarts
        assert got.history.size == want.history.size
        assert abs(got.final_true_residual - want.final_true_residual) <= HIST_TOL * r0
    else:
        assert abs(got.iter_count - want.iter_count) <= max(2, 0.05 * want.iter_count)


def _matrix(name, g):
    if name == "hpcg16":
        return matgen.hpcg(16)
    if name == "hpcg32":
        return matgen.hpcg(32)
    return g["rp"], g["col"], g["val"]


def _keys(g):
    return sorted(k[:-len("__history")] for k in g.files if k.endswith("__history"))


CASES = [(n, k) for n in ("fdm2d16", "band_klein", "hpcg16", "hpcg32", "anderson_12_10_8", "anderson_dd_12_10_8")
         for k in _keys(golden(n))]


@pytest.mark.parametrize("name,key", CASES)
def test_solve_matches_reference_fixture(ctx, name, key):
    g = golden(name)
    rp, col, val = _matrix(name, g)
    method, pre = key.split("__")
    got = host.solve(ctx, method, pre, crs=(rp, col, val))
    stable = check_against_fixture(got, g, key)
    if stable and got.converged:
        x_ref = g[key + "__x"]
        assert np.max(np.abs(got.x_star - x_ref)) <= 1e-9 * max(np.max(np.abs(x_ref)), 1.0)
    assert got.launches > 0


SCALE_CASES = [(n, k) for n in ("fdm2d16_scale", "anderson_dd_12_10_8_scale") for k in _keys(golden(n))]


@pytest.mark.parametrize("name,key", SCALE_CASES)
def test_scaled_solve_matches_reference_fixture(ctx, name, key):
    """-scale 1 (preprocessing.hpp:39-50) through the device path against the compiled reference."""
    g = golden(name)
    method, pre = key.split("__")
    got = host.solve(ctx, method, pre, crs=(g["rp"], g["col"], g["val"]), num_scale=True)
    stable = check_against_fixture(got, g, key)
    if stable and got.converged:
        x_ref = g[key + "__x"]
        assert np.max(np.abs(got.x_star - x_ref)) <= 1e-9 * max(np.max(np.abs(x_ref)), 1.0)
    # the same system, scaled in numpy and handed to the oracle unscaled-API: identical bar
    val_s, sc = port.scale_symmetric(g["rp"], g["col"], g["val"])
    n = len(g["rp"]) - 1
    want = port.solve(g["rp"], g["col"], val_s, method, pre, b=sc * np.ones(n), x0=np.full(n, 0.1))
    check(got, want, exact_count=False)


@pytest.mark.parametrize("method,pre", [("cg", "none"), ("cg", "j"), ("bi", "none"), ("bi", "j"),
                                        ("j", "none"), ("gs", "none"), ("sgs", "none"), ("gm", "none"),
                                        ("gm", "j")])
def test_reference_3x3_solves(ctx, method, pre):
    # tests/test_solvers.cpp:49-91,158-192 (GMRES is disabled there, :187-189; it passes here)
    rp, col, val = i32(0, 2, 5, 7), i32(0, 1, 0, 1, 2, 1, 2), f64(2, -1, -1, 2, -1, -1, 2)
    r = host.solve(ctx, method, pre, crs=(rp, col, val), b=f64(0, 0, 4), x0=f64(0, 0, 0))
    assert r.converged and np.max(np.abs(r.x_star - f64(1, 2, 3))) <= 1e-7


def test_reference_3x3_bicgstab_jacobi_diag10(ctx):
    # tests/test_solvers.cpp:93-141
    rp, col, val = i32(0, 2, 5, 7), i32(0, 1, 0, 1, 2, 1, 2), f64(10, -1, -1, 10, -1, -1, 10)
    xt = f64(1, 2, 3)
    r = host.solve(ctx, "bi", "j", crs=(rp, col, val), b=port.spmv(rp, col, val, xt), x0=f64(0, 0, 0))
    assert r.converged and np.max(np.abs(r.x_star - xt)) <= 1e-7


@pytest.mark.parametrize("method,pre,restart", [("cg", "sgs", 10), ("bi", "j", 10), ("cg", "none", 10),
                                                ("gm", "ilu0", 10), ("gm", "sgs", 25), ("bi", "ilu0", 10),
                                                ("cg", "2st", 10), ("gm", "s2st", 10)])
def test_solve_matches_oracle_hpcg_nonuniform(ctx, method, pre, restart):
    """Seeded inputs, non-cubic grid, random rhs / initial guess: GPU vs oracle run here."""
    rp, col, val = matgen.hpcg(20, 14, 11)
    rng = np.random.default_rng(21)
    n = len(rp) - 1
    b, x0 = rng.uniform(0.5, 1.5, n), rng.uniform(-0.1, 0.1, n)
    for tol, exact in ((1e-10, True), (0.0, False)):      # 0.0 = the shipped TOL (1e-14)
        want = port.solve(rp, col, val, method, pre, restart_len=restart, b=b, x0=x0, tol=tol)
        got = host.solve(ctx, method, pre, crs=(rp, col, val), restart_len=restart, b=b, x0=x0, tol=tol)
        check(got, want, exact)


def test_stationary_sweeps_match_oracle(ctx):
    rp, col, val = matgen.hpcg(12)
    for method in ("j", "gs", "sgs"):
        want = port.solve(rp, col, val, method, "none")
        got = host.solve(ctx, method, "none", crs=(rp, col, val))
        # every vector of a stationary sweep is bit-identical to the oracle's; only the norm's
        # reduction order differs (1 ulp), so the count matches even at TOL = 1e-14
        check(got, want, True)
        assert np.array_equal(got.x_star, want.x_star)


def test_device_generated_matrix_equals_uploaded(ctx):
    """`HPCG-<n>` names are generated on the device for methods that need no factors; the
    history must be bit-identical to the same solve on the uploaded host CRS."""
    rp, col, val = matgen.hpcg(24)
    for method, pre in (("cg", "none"), ("bi", "j"), ("j", "none")):
        a = host.solve(ctx, method, pre, crs=(rp, col, val), max_iters=60)
        b = host.solve(ctx, method, pre, matrix_name="HPCG-24", max_iters=60, want_x=False)
        assert a.iter_count == b.iter_count and np.array_equal(a.history, b.history)


def test_bench_session_iterate_copy_matches_solve(ctx):
    """The iterate a CG bench session copies out after its warm-up and timed steps (bench.py --dump-outputs) is the
    x_star of a solve stopped after as many iterations, and the session's residual norms are that solve's."""
    rp, col, val = matgen.hpcg(16)
    n = rp.size - 1
    want = host.solve(ctx, "cg", "j", crs=(rp, col, val), max_iters=8)
    sess = host.BenchSession(ctx, "HPCG-16", "cg", "j")
    try:
        sess.prepare(3)
        sess.run(5)
        x = ctx.alloc(n)
        sess.copy_x(x)
        got = ctx.download(x, n)
        ctx.free(x)
        hist = sess.history(16)
    finally:
        sess.close()
    assert hist.size == want.history.size == 9
    assert np.max(np.abs(hist - want.history)) <= HIST_TOL * want.history[0]
    assert np.max(np.abs(got - want.x_star)) <= 1e-12 * np.max(np.abs(want.x_star))


def test_run_to_run_determinism(ctx):
    rp, col, val = matgen.hpcg(20)
    for method, pre in (("cg", "sgs"), ("gm", "ilu0"), ("bi", "j")):
        a = host.solve(ctx, method, pre, crs=(rp, col, val))
        b = host.solve(ctx, method, pre, crs=(rp, col, val))
        assert np.array_equal(a.history, b.history) and np.array_equal(a.x_star, b.x_star)


def test_size_independent_properties_at_scale(ctx):
    """HPCG-128 (BASELINE config 1/2 size), no oracle run: (a) the final TRUE residual of the
    returned x_star, recomputed by the harness, is below the stopping threshold region;
    (b) CG on an SPD matrix: the recurrence residual tracks the true residual;
    (c) the published reference numbers for this size (BASELINE.md section 2)."""
    r = host.solve(ctx, "cg", "none", matrix_name="HPCG-128", want_x=False)
    assert abs(r.history[0] - 1.4148190838408811e+03) <= 1e-10 * r.history[0]
    assert abs(r.history[1] - 9.4222420031314541e+03) <= 1e-10 * r.history[0]
    assert abs(r.history[100] - 4.1442144142479105e+00) <= 1e-10 * r.history[0]
    # reference: 290 / 290 / 275 / 279 iterations at 1 / 2 / 4 / 8 OpenMP threads (its own dot-product
    # order decides, F7); the device's tree reductions are more accurate and converge a little earlier
    assert r.converged and 230 <= r.iter_count <= 300
    res3 = int(np.argmax(r.history / r.history[0] < 1e-3))
    res6 = int(np.argmax(r.history / r.history[0] < 1e-6))
    assert (res3, res6) == (107, 150)
    assert r.final_true_residual <= 1e-11 * r.history[0]     # true residual of x_star, recomputed
    b = host.solve(ctx, "bi", "j", matrix_name="HPCG-128", want_x=False)
    assert abs(b.history[1] - 2.4190103171406172e+03) <= 1e-10 * b.history[0]
    assert b.converged and 150 <= b.iter_count <= 230     # reference: 189 at 8 threads; same caveat
    j = host.solve(ctx, "j", "none", matrix_name="HPCG-128", want_x=False)
    assert not j.converged and j.iter_count == 1000
    assert abs(j.history[1000] - 5.8007937268987325e+02) <= 1e-10 * j.history[0]


def test_two_gpu_partition_matches_single_gpu():
    """Needs >= 2 GPUs (skipped on the single-GPU box): tools/dist_check.py under torchrun."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533", "tools/dist_check.py", "40"],
                         cwd=root, capture_output=True, text=True, timeout=600)
    assert "DIST_CHECK PASS" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


def test_factors_without_natural_crs_give_the_same_history(ctx):
    """factor_keep_crs = 0 (what the C++ host selects for a Krylov method with a gs / sgs / ilu0 preconditioner):
    the factors keep only their level-ordered copy; histories are bit-identical, and an entry point that needs the
    factor's CRS arrays fails loudly instead of reading freed memory."""
    for method, pre in (("cg", "sgs"), ("gm", "ilu0"), ("bi", "gs")):
        a = host.solve(ctx, method, pre, matrix_name="HPCG-24", want_x=False, max_iters=60)
        assert a.iter_count > 0
    # the host turns the option on by itself; compare against an explicit split with the arrays kept
    A = ctx.generate_hpcg(24)
    n = A.info()["n_rows"]
    D = ctx.alloc(n)
    ctx.call("bis_matrix_extract_diagonal", A.h, D, None)
    bh = np.random.default_rng(11).uniform(-1.0, 1.0, n)
    out = {}
    for keep in (1, 0):
        ctx.set_option("factor_keep_crs", keep)
        try:
            L, U = ctx.split_triangular(A)
        finally:
            ctx.set_option("factor_keep_crs", 1)
        b, x, y = ctx.upload(bh), ctx.alloc(n), ctx.alloc(n)
        ctx.call("bis_sptrsv", L.h, x, D, b)
        ctx.call("bis_bsptrsv", U.h, y, D, b)
        ctx.sync()
        out[keep] = (ctx.download(x, n), ctx.download(y, n))
        if keep == 0:
            with pytest.raises(capi.BisError):
                ctx.call("bis_spmv", L.h, b, x)
        for m in (L, U):
            m.free()
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
