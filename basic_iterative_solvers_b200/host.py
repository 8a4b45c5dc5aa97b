"""ctypes binding of the HOST library (host/host_capi.cpp -> lib/libbis_host.so).

libbis_host.so holds the reference-shaped Solver / solver_harness / methods
stack (C++), which drives the device through the C-ABI of libbis_b200.so.  This
module only marshals arguments: the iteration loop itself runs in C++.
No CPU fallback: `solve` needs a capi.Context, i.e. a B200.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

from . import capi

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libbis_host.so")
CLI_PATH = os.path.join(HERE, "lib", "bis")

# SolverType / PrecondType of host/common.hpp (= reference common.hpp:38-56)
METHOD = {"j": 0, "gs": 1, "sgs": 2, "gm": 3, "cg": 4, "bi": 5}
PRECOND = capi.PRECOND
MAX_ITERS = 1000

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    capi.load()   # libbis_b200.so first (libbis_host.so links against it via $ORIGIN)
    if not os.path.exists(LIB_PATH):
        raise capi.BisError(f"{LIB_PATH} is missing: run __graft_entry__.build()")
    lib = C.CDLL(LIB_PATH)
    lib.bis_host_last_error.restype = C.c_char_p
    lib.bis_host_parse_cli.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_int)]
    lib.bis_host_factor.argtypes = [C.c_int] + [C.c_void_p] * 3 + [C.c_int] + [C.c_void_p] * 10
    lib.bis_host_matrix_begin.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.bis_host_matrix_fetch.argtypes = [C.c_void_p] * 3
    lib.bis_host_gmres_least_squares.argtypes = [C.c_int, C.c_int] + [C.c_void_p] * 6
    lib.bis_host_gmres_least_squares.restype = None
    lib.bis_host_gmres_update_g.argtypes = [C.c_int, C.c_int] + [C.c_void_p] * 3 + [C.c_double]
    lib.bis_host_gmres_update_g.restype = C.c_double
    lib.bis_host_solve.argtypes = ([C.c_void_p, C.c_char_p, C.c_int] + [C.c_void_p] * 3 + [C.c_int] * 3 +
                                   [C.c_void_p] * 2 + [C.c_int, C.c_double, C.c_int, C.c_int] + [C.c_void_p] * 5)
    lib.bis_host_bench_open.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int]
    lib.bis_host_bench_open.restype = C.c_void_p
    lib.bis_host_bench_close.argtypes = [C.c_void_p]
    lib.bis_host_bench_close.restype = None
    lib.bis_host_bench_e2e.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 5
    lib.bis_host_bench_prepare.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    lib.bis_host_bench_setup_ms.argtypes = [C.c_void_p]
    lib.bis_host_bench_setup_ms.restype = C.c_double
    lib.bis_host_bench_history.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    lib.bis_host_bench_run.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    lib.bis_host_bench_copy_x.argtypes = [C.c_void_p, C.c_void_p]
    _lib = lib
    return lib


def _err() -> str:
    return load().bis_host_last_error().decode(errors="replace")


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def parse_cli(argv: list[str]) -> dict:
    """parse_cli of host/utilities.hpp (reference utilities/utilities.hpp:12-108)."""
    lib = load()
    arr = (C.c_char_p * len(argv))(*[a.encode() for a in argv])
    out = (C.c_int * 4)()
    if lib.bis_host_parse_cli(len(argv), arr, out) != 0:
        raise capi.BisError(_err())
    inv_m = {v: k for k, v in METHOD.items()}
    inv_p = {v: k for k, v in PRECOND.items()}
    return {"method": inv_m[out[0]], "precond": inv_p[out[1]], "restart_length": out[2],
            "num_scale": bool(out[3])}


@dataclass
class Factors:
    l_rp: np.ndarray
    l_col: np.ndarray
    l_val: np.ndarray
    u_rp: np.ndarray
    u_col: np.ndarray
    u_val: np.ndarray
    A_D: np.ndarray
    A_D_inv: np.ndarray
    L_D: np.ndarray
    U_D: np.ndarray


def factor(rp, col, val, precond="none") -> Factors:
    """factor_LU of host/lu_factors.hpp (reference LU_factors.hpp:900-934)."""
    lib = load()
    rp = np.ascontiguousarray(rp, np.int32)
    col = np.ascontiguousarray(col, np.int32)
    val = np.ascontiguousarray(val, np.float64)
    n = rp.size - 1
    l_rp, u_rp = np.zeros(n + 1, np.int32), np.zeros(n + 1, np.int32)
    if lib.bis_host_factor(n, _p(rp), _p(col), _p(val), PRECOND[precond], _p(l_rp), None, None,
                           _p(u_rp), None, None, None, None, None, None) != 0:
        raise capi.BisError(_err())
    nl, nu = int(l_rp[n]), int(u_rp[n])
    f = Factors(l_rp, np.zeros(max(nl, 1), np.int32), np.zeros(max(nl, 1)), u_rp,
                np.zeros(max(nu, 1), np.int32), np.zeros(max(nu, 1)),
                np.zeros(n), np.zeros(n), np.zeros(n), np.zeros(n))
    if lib.bis_host_factor(n, _p(rp), _p(col), _p(val), PRECOND[precond], _p(f.l_rp), _p(f.l_col),
                           _p(f.l_val), _p(f.u_rp), _p(f.u_col), _p(f.u_val), _p(f.A_D),
                           _p(f.A_D_inv), _p(f.L_D), _p(f.U_D)) != 0:
        raise capi.BisError(_err())
    f.l_col, f.l_val = f.l_col[:nl], f.l_val[:nl]
    f.u_col, f.u_val = f.u_col[:nu], f.u_val[:nu]
    return f


def matrix(name: str):
    """CRS of a named matrix: .mtx path, HPCG-<n>, HPCG-<nx>-<ny>-<nz>, Anderson,Lx=..,..."""
    lib = load()
    n, nnz = C.c_int(0), C.c_int(0)
    if lib.bis_host_matrix_begin(name.encode(), C.byref(n), C.byref(nnz)) != 0:
        raise capi.BisError(_err())
    rp = np.zeros(n.value + 1, np.int32)
    col = np.zeros(max(nnz.value, 1), np.int32)
    val = np.zeros(max(nnz.value, 1))
    lib.bis_host_matrix_fetch(_p(rp), _p(col), _p(val))
    return rp, col[:nnz.value], val[:nnz.value]


def gmres_least_squares(k, m, J, H, H_tmp, Q, Q_tmp, R):
    load().bis_host_gmres_least_squares(k, m, _p(J), _p(H), _p(H_tmp), _p(Q), _p(Q_tmp), _p(R))


def gmres_update_g(k, m, Q, g, g_tmp, beta) -> float:
    return load().bis_host_gmres_update_g(k, m, _p(Q), _p(g), _p(g_tmp), float(beta))


@dataclass
class SolveResult:
    history: np.ndarray          # collected_residual_norms[0:count]
    final_true_residual: float   # ||b - A x_star|| from save_x_star
    iter_count: int
    converged: bool
    restarts: int
    stopping_criteria: float
    x_star: np.ndarray | None
    iter_time: np.ndarray        # harness per-iteration seconds (time_per_iteration[1:count+1])
    solve_time: float
    preprocessing_time: float
    mean_iter_time: float
    launches: int


def solve(ctx: capi.Context, method: str, precond: str = "none", *, crs=None, matrix_name=None,
          restart_len: int = 10, b=None, x0=None, max_iters: int = 0, tol: float = 0.0,
          quiet: bool = True, want_x: bool = True, num_scale: bool = False) -> SolveResult:
    """preprocessing() + solve() of the host stack on the device behind `ctx`.

    crs = (row_ptr, col, val) host arrays, or matrix_name = generator / file
    name (device-side generation when no triangular factors are needed).
    """
    lib = load()
    hist = np.zeros(2 * MAX_ITERS)
    itime = np.zeros(2 * MAX_ITERS)
    oi = (C.c_int * 8)()
    od = (C.c_double * 8)()
    if crs is not None:
        rp = np.ascontiguousarray(crs[0], np.int32)
        col = np.ascontiguousarray(crs[1], np.int32)
        val = np.ascontiguousarray(crs[2], np.float64)
        n = rp.size - 1
        name = None
    else:
        if matrix_name is None:
            raise ValueError("solve: give crs= or matrix_name=")
        rp = col = val = None
        n = 0
        name = matrix_name.encode()
    bb = None if b is None else np.ascontiguousarray(b, np.float64)
    xx = None if x0 is None else np.ascontiguousarray(x0, np.float64)
    # x_star length: local rows; for a named matrix ask for it afterwards
    xs = np.zeros(n) if (want_x and crs is not None) else None
    rc = lib.bis_host_solve(ctx.h, name, n, _p(rp), _p(col), _p(val), METHOD[method], PRECOND[precond],
                            restart_len, _p(bb), _p(xx), int(max_iters), float(tol), int(quiet), int(num_scale),
                            _p(hist), _p(itime), _p(xs), oi, od)
    if rc != 0:
        raise capi.BisError(_err())
    cnt = int(oi[1])
    return SolveResult(hist[:cnt].copy(), float(od[1]), int(oi[0]), bool(oi[2]), int(oi[3]),
                       float(od[0]), xs, itime[1:cnt + 1].copy(), float(od[2]), float(od[3]),
                       float(od[4]), int(oi[4]))


def harness_trace(run_ahead: bool, max_iters: int, tol: float, decay: float):
    """solve() of host/solver_harness.hpp on a device-free recording solver (CPU-only test aid)."""
    lib = load()
    lib.bis_host_harness_trace.argtypes = [C.c_int, C.c_int, C.c_double, C.c_double, C.c_char_p, C.c_int, C.c_void_p]
    buf = C.create_string_buffer(1 << 16)
    out = (C.c_int * 4)()
    if lib.bis_host_harness_trace(int(run_ahead), max_iters, tol, decay, buf, len(buf), out) != 0:
        raise capi.BisError(_err())
    return buf.value.decode(), {"iter_count": out[0], "iterates": out[1], "converged": bool(out[2]), "history": out[3]}


class BenchSession:
    """Measurement session of bench.py (host/host_capi.cpp, "measurement sessions")."""

    def __init__(self, ctx: capi.Context, matrix_name: str, method: str, precond: str = "none",
                 restart_len: int = 10):
        self.lib = load()
        self.h = self.lib.bis_host_bench_open(ctx.h, matrix_name.encode(), METHOD[method], PRECOND[precond],
                                              restart_len)
        if not self.h:
            raise capi.BisError(_err())

    @staticmethod
    def _info(arr):
        return dict(zip(("n_rows", "n_rows_global", "nnz", "nnz_global", "rp_bytes"), (int(v) for v in arr[:5])))

    def e2e(self, steps: int, b_ptr: int | None, x0_ptr: int | None, x_out_ptr: int | None):
        out = (C.c_double * 8)()
        info = (C.c_int64 * 8)()
        if self.lib.bis_host_bench_e2e(self.h, steps, b_ptr, x0_ptr, x_out_ptr, out, info) != 0:
            raise capi.BisError(_err())
        return {"wall_ms": out[0], "iters": int(out[1]), "launches": int(out[2]), "res_last": out[3],
                "res0": out[4], "res_true": out[5],
                "breakdown_ms": {"allocate_init_upload": out[6], "r0_and_factor": out[7],
                                 "iterations": info[6] / 1e3, "x_star_download": info[7] / 1e3},
                **self._info(info)}

    def setup_ms(self) -> float:
        """Wall time of the last matrix set-up (generation, SpMV tile format, order table)."""
        return float(self.lib.bis_host_bench_setup_ms(self.h))

    def history(self, cap: int = 64) -> np.ndarray:
        """First residual norms of the session's current solver."""
        buf = np.zeros(cap)
        n = self.lib.bis_host_bench_history(self.h, _p(buf), cap)
        return buf[:min(n, cap)].copy()

    def prepare(self, warmup: int):
        info = (C.c_int64 * 8)()
        if self.lib.bis_host_bench_prepare(self.h, warmup, info) != 0:
            raise capi.BisError(_err())
        return self._info(info)

    def run(self, steps: int):
        out = (C.c_double * 8)()
        if self.lib.bis_host_bench_run(self.h, steps, out) != 0:
            raise capi.BisError(_err())
        return {"device_ms": out[0], "wall_ms": out[1], "launches": int(out[2]), "res_last": out[3],
                "res0": out[4]}

    def copy_x(self, x_dev: int):
        """Enqueue a copy of the current iterate of a CG session into the device vector x_dev (local rows)."""
        if self.lib.bis_host_bench_copy_x(self.h, x_dev) != 0:
            raise capi.BisError(_err())

    def close(self):
        if self.h:
            self.lib.bis_host_bench_close(self.h)
            self.h = None
