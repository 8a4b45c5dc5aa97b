"""Generate tests/golden/*.npz from the UNMODIFIED reference compiled in the build
container (oracle/_ref/libbis_ref.so, built from /root/reference by oracle/Makefile).

Run from the repo root:  python tests/golden/make_golden.py

The fixtures pin the oracle (oracle/port) and the CUDA path to outputs of the real
reference: residual histories, iteration counts, final true residuals, triangular
factors, ILU(0) factors and kernel outputs.  All golden runs use ONE OpenMP thread
(SURVEY.md F7: the reference's reductions are thread-count dependent); every solve fixture also
records `<key>__noise` = [max_k |r_k(other run) - r_k(1 thread)| / r0 over {8 threads, 4 threads,
pinned-codegen flavour}, min iteration count, max iteration count], i.e. the reference's own
self-noise envelope, which the parity tests use as the floor of their tolerance and the stock
flavour of the build (-O3 -fopenmp, -march=x86-64-v3).  ILU(0) uses factor_ILU0_old
(LU_factors.hpp:320-539): factor_ILU0_new needs the absent SMAX library (SURVEY.md F4).
"""
from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import matgen, refshim  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
REF_DATA = "/root/reference/data/matrices"

SOLVES = [("j", "none"), ("gs", "none"), ("sgs", "none"), ("cg", "none"), ("gm", "none"), ("bi", "none"),
          ("cg", "j"), ("cg", "gs"), ("cg", "sgs"), ("cg", "ilu0"),
          ("gm", "j"), ("gm", "gs"), ("gm", "bgs"), ("gm", "sgs"), ("gm", "ilu0"),
          ("bi", "j"), ("bi", "gs"), ("bi", "bgs"), ("bi", "sgs"), ("bi", "ilu0")]


def solves(rp, col, val, which, restart_len=10, num_scale=False):
    out = {}
    for method, pre in which:
        r = refshim.solve(rp, col, val, method, pre, restart_len=restart_len, threads=1, num_scale=num_scale)
        key = f"{method}__{pre}"
        out[key + "__history"] = r.history
        out[key + "__meta"] = np.array([r.iter_count, int(r.converged), r.restarts], np.int64)
        out[key + "__final"] = np.array([r.final_true_residual, r.stopping_criteria])
        out[key + "__x"] = r.x_star
        # The reference's OWN self-noise envelope (SURVEY.md F7): the same solve at 8 and 4
        # OpenMP threads and with the pinned-codegen flavour, against the 1-thread run above.
        noise, its_lo, its_hi = 0.0, r.iter_count, r.iter_count
        for thr, det in ((8, False), (4, False), (1, True)):
            q = refshim.solve(rp, col, val, method, pre, restart_len=restart_len, threads=thr, det=det,
                              num_scale=num_scale)
            k = min(q.history.size, r.history.size)
            with np.errstate(invalid="ignore"):
                dmax = np.nanmax(np.abs(q.history[:k] - r.history[:k])) / r.history[0]
            noise = max(noise, float(dmax))
            its_lo, its_hi = min(its_lo, q.iter_count), max(its_hi, q.iter_count)
        refshim.load().ref_omp_set_threads(1)
        out[key + "__noise"] = np.array([noise, its_lo, its_hi])
        print(f"  {key:14s} its={r.iter_count:4d} conv={int(r.converged)} restarts={r.restarts} "
              f"r0={r.history[0]:.16e} final={r.final_true_residual:.3e} self-noise={noise:.1e} "
              f"its in [{its_lo},{its_hi}]")
    return out


def kernels(rp, col, val, seed):
    """Kernel-level outputs of the reference on seeded inputs."""
    rng = np.random.default_rng(seed)
    n = rp.size - 1
    x = rng.uniform(-1.0, 1.0, n)
    v = rng.uniform(-1.0, 1.0, n)
    out = {"x": x, "v": v}
    out["spmv"] = refshim.spmv(rp, col, val, x)
    fac = refshim.factor(rp, col, val, "sgs")
    for k in ("l_rp", "l_col", "l_val", "u_rp", "u_col", "u_val", "A_D", "A_D_inv"):
        out["split__" + k] = getattr(fac, k)
    out["sptrsv"] = refshim.sptrsv(fac.l_rp, fac.l_col, fac.l_val, fac.A_D, x)
    out["bsptrsv"] = refshim.sptrsv(fac.u_rp, fac.u_col, fac.u_val, fac.A_D, x, backward=True)
    out["sptrsv_inplace"] = refshim.sptrsv_inplace(fac.l_rp, fac.l_col, fac.l_val, fac.A_D, x)
    for pre in ("none", "j", "gs", "bgs", "sgs"):
        out["precond__" + pre] = refshim.apply_preconditioner(pre, fac, x)
    ilu = refshim.factor(rp, col, val, "ilu0", ilu0_old=True)
    for k in ("l_rp", "l_col", "l_val", "u_rp", "u_col", "u_val", "L_D", "U_D"):
        out["ilu0__" + k] = getattr(ilu, k)
    out["precond__ilu0"] = refshim.apply_preconditioner("ilu0", ilu, x)
    lib = refshim.load()
    for name in ("subtract_vectors", "sum_vectors", "elemwise_mult_vectors", "elemwise_div_vectors"):
        o = np.zeros(n)
        getattr(lib, "ref_" + name)(o, x, v + 2.0, n, 0.37)
        out[name] = o
    o = np.zeros(n)
    lib.ref_scale(o, x, -1.25, n)
    out["scale"] = o
    out["dot"] = np.array([lib.ref_dot(x, v, n)])
    out["norm"] = np.array([lib.ref_euclidean_vec_norm(x, n)])
    xn = refshim.spmv(rp, col, val, x)
    lib.ref_normalize_x(xn, x, fac.A_D, v, n)
    out["normalize_x"] = xn
    return out


def main():
    assert refshim.available(), "build oracle/_ref first: make -C oracle ref"
    refshim.load().ref_omp_set_threads(1)

    for fname, key in (("FDM-2d-16.mtx", "fdm2d16"), ("matrix_band_klein.mtx", "band_klein")):
        print(key)
        rp, col, val = refshim.read_mtx(os.path.join(REF_DATA, fname))
        d = {"rp": rp, "col": col, "val": val}
        d.update(solves(rp, col, val, SOLVES))
        d.update({"k__" + k: v for k, v in kernels(rp, col, val, 7).items()})
        np.savez_compressed(os.path.join(OUT, key + ".npz"), **d)

    print("hpcg16")
    rp, col, val = matgen.hpcg(16)
    d = solves(rp, col, val, SOLVES)
    d.update({"k__" + k: v for k, v in kernels(rp, col, val, 11).items()
              if not k.startswith(("split__", "ilu0__l_", "ilu0__u_r", "ilu0__u_c"))})
    np.savez_compressed(os.path.join(OUT, "hpcg16.npz"), **d)

    print("hpcg32 (headline configs at reduced size)")
    rp, col, val = matgen.hpcg(32)
    d = solves(rp, col, val, [("cg", "none"), ("cg", "sgs"), ("bi", "j"), ("gm", "sgs")])
    # histories only (x_star of 32768 rows x 4 is small enough too)
    np.savez_compressed(os.path.join(OUT, "hpcg32.npz"), **d)

    print("anderson 12x10x8 ranpot=5 seed=1 open BC (config 4 at reduced size)")
    rp, col, val = matgen.anderson(12, 10, 8, ranpot=5.0, t=1.0, seed=1, periodic=False)
    d = {"rp": rp.astype(np.int32), "col": col, "val": val}
    d.update(solves(rp, col, val, [("gm", "ilu0"), ("gm", "j"), ("bi", "ilu0")]))
    np.savez_compressed(os.path.join(OUT, "anderson_12_10_8.npz"), **d)

    # diagonally dominant Anderson (ranpot shifts the spectrum): a well-conditioned ILU(0) case
    print("anderson-dd 12x10x8 (diagonal + 8)")
    val2 = val.copy()
    n = rp.size - 1
    rows = np.repeat(np.arange(n), np.diff(rp))
    val2[rows == col] += 8.0
    d = {"rp": rp.astype(np.int32), "col": col, "val": val2}
    d.update(solves(rp, col, val2, [("gm", "ilu0"), ("cg", "ilu0"), ("bi", "ilu0")]))
    np.savez_compressed(os.path.join(OUT, "anderson_dd_12_10_8.npz"), **d)


def scale_fixtures():
    """-scale 1 (preprocessing.hpp:39-50): the reference solves D^-1/2 A D^-1/2 x' = D^-1/2 b."""
    assert refshim.available(), "build oracle/_ref first: make -C oracle ref"
    refshim.load().ref_omp_set_threads(1)
    print("fdm2d16, -scale 1")
    rp, col, val = refshim.read_mtx(os.path.join(REF_DATA, "FDM-2d-16.mtx"))
    d = {"rp": rp, "col": col, "val": val}
    d.update(solves(rp, col, val, [("cg", "none"), ("cg", "j"), ("cg", "sgs"), ("gm", "ilu0"), ("bi", "j"),
                                   ("j", "none"), ("sgs", "none")], num_scale=True))
    np.savez_compressed(os.path.join(OUT, "fdm2d16_scale.npz"), **d)
    print("anderson-dd 12x10x8, -scale 1 (non-constant diagonal)")
    rp, col, val = matgen.anderson(12, 10, 8, ranpot=5.0, t=1.0, seed=1, periodic=False)
    val2 = val.copy()
    rows = np.repeat(np.arange(rp.size - 1), np.diff(rp))
    val2[rows == col] += 8.0
    d = {"rp": rp.astype(np.int32), "col": col, "val": val2}
    d.update(solves(rp, col, val2, [("cg", "none"), ("gm", "ilu0"), ("bi", "sgs")], num_scale=True))
    np.savez_compressed(os.path.join(OUT, "anderson_dd_12_10_8_scale.npz"), **d)


RANDOM_SOLVES = [("cg", "sgs"), ("bi", "ilu0"), ("gm", "ilu0"), ("sgs", "none")]


def random_system(n=300, seed=3):
    """Symmetric, strictly diagonally dominant matrix with a random sparsity pattern (3 % fill), and a vector x."""
    rng = np.random.default_rng(seed)
    dense = (rng.random((n, n)) < 0.03) * rng.uniform(-1, 1, (n, n))
    dense = dense + dense.T
    np.fill_diagonal(dense, np.abs(dense).sum(axis=1) + 1.0)
    rows, cols = np.nonzero(dense)
    rp = np.zeros(n + 1, np.int32)
    np.add.at(rp, rows + 1, 1)
    rp = np.cumsum(rp).astype(np.int32)
    return rp, cols.astype(np.int32), dense[rows, cols], rng.uniform(-1, 1, n)


def random_fixture():
    """random300.npz: ILU(0) factors, SGS and ILU(0) preconditioner outputs and four whole solves on random_system().
    Written from the compiled reference when oracle/_ref is built, otherwise from the oracle (oracle/port, which
    matches the reference bit for bit on the fixtures above); `source` records which.

        python tests/golden/make_golden.py random300
    """
    from oracle import port
    ref = refshim.available()
    if ref:
        refshim.load().ref_omp_set_threads(1)
    impl = refshim if ref else port
    rp, col, val, x = random_system()
    d = {"source": np.array(["reference" if ref else "oracle"]), "rp": rp, "col": col, "val": val, "x": x}
    ilu = impl.factor(rp, col, val, "ilu0")
    for k in ("l_rp", "l_col", "l_val", "u_rp", "u_col", "u_val", "L_D", "U_D"):
        d["ilu0__" + k] = getattr(ilu, k)
    d["precond__ilu0"] = impl.apply_preconditioner("ilu0", ilu, x)
    d["precond__sgs"] = impl.apply_preconditioner("sgs", impl.factor(rp, col, val, "sgs"), x)
    for method, pre in RANDOM_SOLVES:
        r = refshim.solve(rp, col, val, method, pre, threads=1) if ref else port.solve(rp, col, val, method, pre)
        d[f"{method}__{pre}__history"] = r.history
        d[f"{method}__{pre}__meta"] = np.array([r.iter_count, int(r.converged), r.restarts], np.int64)
        print(f"  {method}__{pre}: its={r.iter_count} conv={int(r.converged)} r0={r.history[0]:.6e}")
    np.savez_compressed(os.path.join(OUT, "random300.npz"), **d)
    print(f"random300.npz written from the {d['source'][0]}")


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "random300":
    random_fixture()
    raise SystemExit(0)

if __name__ == "__main__" and not (len(sys.argv) > 1 and sys.argv[1] == "twostage"):
    if len(sys.argv) > 1 and sys.argv[1] == "scale":
        scale_fixtures()
        raise SystemExit(0)
    main()


def twostage_fixtures():
    """-p 2st / s2st with PRECOND_INNER_ITERS = 1 and 2: the reference fixes the number of inner sweeps at compile
    time (kernels.hpp:321, 0 in its default build), so the fixtures come from the flavours oracle/_ref/libbis_ref_in1.so
    and _in2.so (oracle/Makefile).  Preconditioner applications (bit-exact targets) and whole solves.

        python tests/golden/make_golden.py twostage
    """
    d = {}
    rng = np.random.default_rng(23)
    for name, (rp, col, val) in (("hpcg12", matgen.hpcg(12)), ("hpcg_10_7_5", matgen.hpcg(10, 7, 5))):
        n = rp.size - 1
        x = rng.uniform(-1.0, 1.0, n)
        d[f"{name}__x"] = x
        for inner in (1, 2):
            flav = f"in{inner}"
            assert refshim.available(flav), "build oracle/_ref first: make -C oracle ref"
            refshim.load(flav).ref_omp_set_threads(1)
            fac = refshim.factor(rp, col, val, "sgs", det=flav)
            for pre in ("2st", "s2st"):
                d[f"{name}__in{inner}__precond__{pre}"] = refshim.apply_preconditioner(pre, fac, x, det=flav)
            for method, pre in (("cg", "2st"), ("cg", "s2st"), ("gm", "s2st"), ("bi", "2st")):
                r = refshim.solve(rp, col, val, method, pre, det=flav, threads=1)
                key = f"{name}__in{inner}__{method}__{pre}"
                d[key + "__history"] = r.history
                d[key + "__meta"] = np.array([r.iter_count, int(r.converged), r.restarts], np.int64)
                print(f"  {key}: its={r.iter_count} conv={int(r.converged)} r0={r.history[0]:.6e}")
    np.savez_compressed(os.path.join(OUT, "twostage.npz"), **d)


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "twostage":
    twostage_fixtures()
