"""oracle/port.py -- TEST INFRASTRUCTURE.

ctypes binding of oracle/libbis_oracle.so, the plain-C restatement
(oracle/port/bis_oracle.c).  Same call shapes as oracle/refshim.py so tests
can run either checker on the same inputs.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from .refshim import METHOD, PRECOND, MAX_ITERS, Factors, SolveResult  # noqa: F401

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libbis_oracle.so")

_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")


class _Crs(C.Structure):
    _fields_ = [("n", C.c_int), ("nnz", C.c_int), ("rp", C.c_void_p), ("col", C.c_void_p),
                ("val", C.c_void_p)]


def build() -> None:
    subprocess.check_call(["make", "-s", "-C", HERE, "port"])


_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    src = os.path.join(HERE, "port", "bis_oracle.c")
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(src):
        build()
    lib = C.CDLL(LIB)
    lib.o_spmv.argtypes = [C.c_int, _ip, _ip, _dp, _dp, _dp]
    lib.o_sptrsv.argtypes = [C.c_int, _ip, _ip, _dp, _dp, _dp, _dp]
    lib.o_bsptrsv.argtypes = [C.c_int, _ip, _ip, _dp, _dp, _dp, _dp]
    for f in ("o_subtract_vectors", "o_sum_vectors", "o_elemwise_mult_vectors",
              "o_elemwise_div_vectors"):
        getattr(lib, f).argtypes = [_dp, _dp, _dp, C.c_int, C.c_double]
    lib.o_scale.argtypes = [_dp, _dp, C.c_double, C.c_int]
    lib.o_dot.argtypes = [_dp, _dp, C.c_int]
    lib.o_dot.restype = C.c_double
    lib.o_euclidean_vec_norm.argtypes = [_dp, C.c_int]
    lib.o_euclidean_vec_norm.restype = C.c_double
    lib.o_normalize_x.argtypes = [_dp, _dp, _dp, _dp, C.c_int]
    lib.o_apply_preconditioner.argtypes = [C.c_int, C.c_int, C.POINTER(_Crs), C.POINTER(_Crs)] + [_dp] * 8
    lib.o_split_strict.argtypes = [C.c_int, _ip, _ip, _dp] + [C.c_void_p] * 8
    lib.o_ilu0.argtypes = [C.c_int, _ip, _ip, _dp, _ip, _ip, _dp, _dp, _ip, _ip, _dp, _dp]
    lib.o_gmres_least_squares.argtypes = [C.c_int, C.c_int] + [_dp] * 6
    lib.o_gmres_update_g.argtypes = [C.c_int, C.c_int, _dp, _dp, _dp, C.c_double]
    lib.o_gmres_update_g.restype = C.c_double
    lib.o_solve.argtypes = [C.c_int, _ip, _ip, _dp, C.c_int, C.c_int, C.c_int, C.c_void_p,
                            C.c_void_p, _dp, _dp, _ip, _dp]
    lib.o_solve.restype = C.c_int
    lib.o_set_params.argtypes = [C.c_double, C.c_int]
    _lib = lib
    return lib


def _crs(rp, col, val):
    rp = np.ascontiguousarray(rp, dtype=np.int32)
    col = np.ascontiguousarray(col, dtype=np.int32)
    val = np.ascontiguousarray(val, dtype=np.float64)
    if col.size == 0:
        col = np.zeros(1, np.int32)
        val = np.zeros(1, np.float64)
    return rp, col, val


def spmv(rp, col, val, x):
    lib = load()
    rp, col, val = _crs(rp, col, val)
    y = np.zeros(rp.size - 1)
    lib.o_spmv(rp.size - 1, rp, col, val, np.ascontiguousarray(x, dtype=np.float64), y)
    return y


def sptrsv(rp, col, val, D, b, backward=False, x_init=None):
    lib = load()
    rp, col, val = _crs(rp, col, val)
    n = rp.size - 1
    x = np.zeros(n) if x_init is None else np.array(x_init, dtype=np.float64)
    (lib.o_bsptrsv if backward else lib.o_sptrsv)(n, rp, col, val, x, np.ascontiguousarray(D),
                                                  np.ascontiguousarray(b))
    return x


def sptrsv_inplace(rp, col, val, D, xb, backward=False):
    lib = load()
    rp, col, val = _crs(rp, col, val)
    x = np.array(xb, dtype=np.float64)
    (lib.o_bsptrsv if backward else lib.o_sptrsv)(rp.size - 1, rp, col, val, x,
                                                  np.ascontiguousarray(D), x)
    return x


# ---- slab-wise application ----------------------------------------------------------------------------
# A matrix whose nonzeros do not fit the oracle's int row_ptr is applied one row slab [rb, re) at a time.  A
# slab comes as CRS with a row_ptr that starts at 0 (int32 for any slab of moderate height) and its columns
# rebased to rb.  The unchanged C loops then run on views of the full vectors that start at row rb (x[rb:],
# y[rb:], D[rb:], b[rb:]): a negative rebased column reads an earlier row through the view, and every row gets
# the products, sums and roundings of the whole-matrix call.  Rebased to its own first row, every interior
# slab of an HPCG grid has the same local structure, so three generated templates (first, interior, last)
# serve the whole matrix.

def rebase(rp, col, val, row_begin):
    """a slab's CRS from matgen (global columns) with its columns made relative to row_begin"""
    rp = np.ascontiguousarray(rp, dtype=np.int32)
    col = np.ascontiguousarray(np.asarray(col, np.int64) - int(row_begin), dtype=np.int32)
    return _crs(rp, col, val)


def split_rebased(rp, col, val):
    """(L, U, diag) of a rebased slab: strictly lower / upper parts as (rp, col, val), entries in storage order
    exactly as o_split_strict keeps them; diag[i] is the last diagonal entry of row i (o_split_strict's A_D)"""
    rp = np.asarray(rp, np.int64)
    m = rp.size - 1
    cnt = np.diff(rp)
    rows = np.repeat(np.arange(m, dtype=np.int64), cnt)
    col = np.asarray(col[:rp[-1]], np.int64)
    val = np.asarray(val[:rp[-1]])
    out = []
    for keep in (col < rows, col > rows):
        t_rp = np.zeros(m + 1, np.int32)
        np.cumsum(np.bincount(rows[keep], minlength=m), out=t_rp[1:])
        out.append(_crs(t_rp, col[keep].astype(np.int32), val[keep]))
    diag = np.zeros(m)
    on = col == rows
    diag[rows[on]] = val[on]
    return out[0], out[1], diag


class GeneratedSlabs:
    """Row slabs of `slab_rows` rows, each generated by gen(row_begin, row_end) -> (rp, col, val)"""

    def __init__(self, gen, n, slab_rows):
        self.gen, self.n = gen, n
        self.bounds = [(rb, min(rb + slab_rows, n)) for rb in range(0, n, slab_rows)]

    def crs(self, rb, re):
        return rebase(*self.gen(rb, re), rb)

    def split(self, rb, re):
        return split_rebased(*self.crs(rb, re))


class TemplatedSlabs:
    """Row slabs of `planes` grid planes of a stencil matrix whose rebased structure and off-diagonal values
    are the same in every interior slab, served from at most three templates generated by gen(row_begin,
    row_end): the first slab, the interior ones and the last.  diagonal(rows), when given, supplies the
    row-dependent diagonal values that are written into a copy of the template."""

    def __init__(self, gen, n, plane, planes, diagonal=None):
        self.n = n
        self.diagonal = diagonal
        self.bounds = [(rb, min(rb + planes * plane, n)) for rb in range(0, n, planes * plane)]
        self._crs, self._split, self._dpos = {}, {}, {}
        for rb, re in self.bounds:
            key = self._key(rb, re)
            if key not in self._crs:
                self._crs[key] = rebase(*gen(rb, re), rb)
                if diagonal is not None:
                    rp, col, _ = self._crs[key]
                    rows = np.repeat(np.arange(re - rb), np.diff(rp))
                    pos = np.flatnonzero(col[:rp[-1]] == rows)
                    assert np.array_equal(rows[pos], np.arange(re - rb)), "one diagonal entry per row"
                    self._dpos[key] = pos

    def _key(self, rb, re):
        return rb == 0, re == self.n, re - rb

    def crs(self, rb, re):
        key = self._key(rb, re)
        if self.diagonal is None:
            return self._crs[key]
        rp, col, val = self._crs[key]
        val = val.copy()
        val[self._dpos[key]] = self.diagonal(np.arange(rb, re, dtype=np.int64))
        return rp, col, val

    def split(self, rb, re):
        if self.diagonal is not None:
            return split_rebased(*self.crs(rb, re))
        key = self._key(rb, re)
        if key not in self._split:
            self._split[key] = split_rebased(*self._crs[key])
        return self._split[key]


def hpcg_slabs(nx, ny, nz, planes):
    from . import matgen
    return TemplatedSlabs(lambda rb, re: matgen.hpcg(nx, ny, nz, rb, re), nx * ny * nz, nx * ny, planes)


def anderson_slabs(lx, ly, lz, planes, ranpot=5.0, t=1.0, seed=1, periodic=False):
    from . import matgen
    return TemplatedSlabs(lambda rb, re: matgen.anderson(lx, ly, lz, ranpot, t, seed, periodic, rb, re),
                          lx * ly * lz, lx * ly, planes, lambda rows: matgen.anderson_diagonal(rows, ranpot, seed))


def spmv_slab_into(rp, col, val, x, y, row_begin):
    """y[row_begin : row_begin + m] = rows of a rebased slab applied to the full x"""
    m = rp.size - 1
    load().o_spmv(m, rp, col, val, x[row_begin:], y[row_begin:row_begin + m])


def spmv_slabwise(slabs, x, threads=None):
    """y = A x slab by slab (slabs: GeneratedSlabs or HpcgSlabs); slabs are independent and the C loop runs
    outside the GIL, so they are spread over threads"""
    from concurrent.futures import ThreadPoolExecutor
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.empty(slabs.n)

    def one(b):
        spmv_slab_into(*slabs.crs(*b), x, y, b[0])

    with ThreadPoolExecutor(threads or os.cpu_count() or 1) as ex:
        list(ex.map(one, slabs.bounds))
    return y


def sptrsv_slab(rp, col, val, x, D, b, row_begin, backward=False):
    """Rows [row_begin, row_begin + m) of o_sptrsv (o_bsptrsv if backward) on the full vectors, in place in x:
    the strictly triangular slab (rp, col, val) has columns rebased to row_begin.  Forward slabs must run in
    ascending order, backward ones in descending order, exactly as the whole-matrix loop visits their rows."""
    lib = load()
    rb = int(row_begin)
    (lib.o_bsptrsv if backward else lib.o_sptrsv)(rp.size - 1, rp, col, val, x[rb:], D[rb:], b[rb:])


def sptrsv_slabwise(slabs, D, b, backward=False):
    """x with D x + T x = b for the strictly lower (upper if backward) part T of the slabbed matrix"""
    x = np.zeros(slabs.n)
    D = np.ascontiguousarray(D, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    for rb, re in (reversed(slabs.bounds) if backward else slabs.bounds):
        L, U, _ = slabs.split(rb, re)
        sptrsv_slab(*(U if backward else L), x, D, b, rb, backward)
    return x


def _vp(a):
    return None if a is None else a.ctypes.data


def factor(rp, col, val, precond="none") -> Factors:
    lib = load()
    rp, col, val = _crs(rp, col, val)
    n = rp.size - 1
    l_rp, u_rp = np.zeros(n + 1, np.int32), np.zeros(n + 1, np.int32)
    lib.o_split_strict(n, rp, col, val, _vp(l_rp), None, None, _vp(u_rp), None, None, None, None)
    nl, nu = int(l_rp[n]), int(u_rp[n])
    f = Factors(l_rp, np.zeros(max(nl, 1), np.int32), np.zeros(max(nl, 1)), u_rp,
                np.zeros(max(nu, 1), np.int32), np.zeros(max(nu, 1)),
                np.ones(n), np.zeros(n), np.ones(n), np.ones(n))
    lib.o_split_strict(n, rp, col, val, _vp(f.l_rp), _vp(f.l_col), _vp(f.l_val), _vp(f.u_rp),
                       _vp(f.u_col), _vp(f.u_val), _vp(f.A_D), _vp(f.A_D_inv))
    if precond == "ilu0":
        lib.o_ilu0(n, rp, col, val, f.l_rp, f.l_col, f.l_val, f.L_D, f.u_rp, f.u_col, f.u_val, f.U_D)
    f.l_col, f.l_val = f.l_col[:nl], f.l_val[:nl]
    f.u_col, f.u_val = f.u_col[:nu], f.u_val[:nu]
    return f


def set_precond_inner_iters(k: int) -> None:
    """PRECOND_INNER_ITERS of the reference (kernels.hpp:321) for the two-stage GS preconditioners."""
    load().o_set_precond_inner_iters(int(k))


def apply_preconditioner(precond, fac: Factors, inp, inplace=False):
    lib = load()
    n = fac.A_D.size
    l = _crs(fac.l_rp, fac.l_col, fac.l_val)
    u = _crs(fac.u_rp, fac.u_col, fac.u_val)
    L = _Crs(n, int(l[0][-1]), l[0].ctypes.data, l[1].ctypes.data, l[2].ctypes.data)
    U = _Crs(n, int(u[0][-1]), u[0].ctypes.data, u[1].ctypes.data, u[2].ctypes.data)
    inp = np.array(inp, dtype=np.float64)
    out = inp if inplace else np.zeros(n)
    tmp, work = np.zeros(n), np.zeros(n)
    lib.o_apply_preconditioner(PRECOND[precond], n, C.byref(L), C.byref(U), fac.A_D, fac.A_D_inv,
                               fac.L_D, fac.U_D, out, inp, tmp, work)
    return out


def solve(rp, col, val, method, precond="none", restart_len=10, b=None, x0=None, tol=0.0,
          max_iters=0) -> SolveResult:
    lib = load()
    lib.o_set_params(float(tol), int(max_iters))
    rp, col, val = _crs(rp, col, val)
    n = rp.size - 1
    hist = np.zeros(2 * MAX_ITERS)
    xs = np.zeros(n)
    oi = np.zeros(4, np.int32)
    od = np.zeros(2)
    bb = None if b is None else np.ascontiguousarray(b, dtype=np.float64)
    xx = None if x0 is None else np.ascontiguousarray(x0, dtype=np.float64)
    rc = lib.o_solve(n, rp, col, val, METHOD[method], PRECOND[precond], restart_len,
                     _vp(bb), _vp(xx), hist, xs, oi, od)
    if rc != 0:
        raise RuntimeError(f"o_solve rc={rc}")
    cnt = int(oi[1])
    return SolveResult(hist[:cnt].copy(), float(od[1]), int(oi[0]), bool(oi[2]), int(oi[3]),
                       float(od[0]), xs, np.zeros(0), 0.0, 0.0, 0.0, 0.0)


def scale_symmetric(rp, col, val):
    """-scale 1 restated in numpy (test infrastructure): extract_scale + scale_mat of the reference
    (utilities/LU_factors.hpp:880-898, preprocessing.hpp:15-24).  Returns (val', s) with
    s[r] = 1 / sqrt(|A[r][r]|) (0.0 for a row without diagonal, solver.hpp:105) and
    val'[k] = val[k] * (s[row] * s[col]), every operation rounded separately as the scalar code does.
    The reference then solves with b' = s * b and -- because init_structs copied x_0 before the scaling
    (preprocessing.hpp:33 vs :48) -- still starts from the UNSCALED initial guess."""
    rp = np.asarray(rp, np.int64)
    col = np.asarray(col, np.int64)
    val = np.asarray(val, np.float64)
    n = rp.size - 1
    rows = np.repeat(np.arange(n), np.diff(rp))
    s = np.zeros(n)
    diag = rows == col
    s[rows[diag]] = 1.0 / np.sqrt(np.abs(val[diag]))      # last match wins, as in the reference's loop
    return val * (s[rows] * s[col]), s
