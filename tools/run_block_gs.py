"""Block Gauss-Seidel / SGS (several right-hand sides, one matrix) against the single-RHS sweeps, on one GPU.

    python tools/run_block_gs.py --out <dir> [--warmup 5] [--steps 50]

One process, one output directory, one JSON file (block_gs.json).  Per matrix (HPCG-128, HPCG-256) and method (gs, sgs)
it runs two rounds, each the single-RHS solve (host.BenchSession) followed by the block solve at k = 1, 2, 4, 8, 16
(host.bench_block), and records per k:
  - block ms/iter, ms/iter per right-hand side and the gain per right-hand side over the single-RHS solve of the same
    round (CUDA events over `steps` iterations after `warmup`, tolerance 0, distinct seeded right-hand sides; column 0
    is b = 1 from INIT_X_VAL, the single-RHS run's system), the median of the two rounds beside each round;
  - the forward block solve alone (bis_block_sptrsv on L, CUDA events over 20 launches) in us per level, next to the
    single-vector dataflow solve (trsv_variant 3) and the stencil wavefront (trsv_variant 5) on the same factor.
It checks itself: the first residuals of block column 0 must be within 1e-10 ||r0|| of the single-RHS run's.
The GPU name and power limit are read in the same run (read-only query).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from basic_iterative_solvers_b200 import capi, host  # noqa: E402

KS = [1, 2, 4, 8, 16]


def gpu_header():
    out = {"gpu": None, "power_limit_w": None}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out = {"gpu": q[0].strip(), "power_limit_w": float(q[1]), "sm_max_mhz": float(q[2])}
    except Exception as e:  # the numbers below are still device-timed; the header says what is missing
        out["header_error"] = repr(e)
    return out


def rhs(n, k, seed):
    B = np.empty((n, k))
    B[:, 0] = 1.0
    rng = np.random.default_rng(seed)
    for j in range(1, k):
        B[:, j] = rng.uniform(-1.0, 1.0, n)
    return B


def time_calls(ctx, fn, reps=20):
    for _ in range(3):
        fn()
    ctx.sync()
    ctx.timer_start()
    for _ in range(reps):
        fn()
    return ctx.timer_stop() / reps


def sweep_per_level(ctx, size):
    """us per level of one forward solve on HPCG-size's L: block at every k, single-vector dataflow and wavefront."""
    A = ctx.generate_hpcg(size)
    L, U = ctx.split_triangular(A)
    n = A.info()["n_rows"]
    D = ctx.alloc(n)
    ctx.call("bis_matrix_extract_diagonal", A.h, D, None)
    x, b = ctx.alloc(n), ctx.alloc(n)
    ctx.call("bis_init_vector", b, 1.0, n)
    out = {}
    for variant, key in ((3, "single_dataflow"), (5, "single_wavefront")):
        ctx.set_option("trsv_variant", variant)
        try:
            out[key] = {"ms": time_calls(ctx, lambda: ctx.call("bis_sptrsv", L.h, x, D, b))}
        except capi.BisError as e:
            out[key] = {"error": str(e)}
        finally:
            ctx.set_option("trsv_variant", 0)
    levels = L.info()["n_levels"]   # read after the dataflow solve: a factor the wavefront serves builds them on demand
    out["n_levels"] = levels
    for key in ("single_dataflow", "single_wavefront"):
        if "ms" in out[key]:
            out[key]["us_per_level"] = out[key]["ms"] * 1e3 / levels
    out["block"] = []
    for k in KS:
        X, Bk = ctx.alloc(n * k), ctx.alloc(n * k)
        ctx.call("bis_init_vector", Bk, 1.0, n * k)
        ms = time_calls(ctx, lambda: ctx.call("bis_block_sptrsv", L.h, k, X, D, Bk, None))
        out["block"].append({"k": k, "ms": ms, "us_per_level": ms * 1e3 / levels, "ms_per_rhs": ms / k})
        ctx.free(X), ctx.free(Bk)
    ctx.free(x), ctx.free(b), ctx.free(D)
    L.free(), U.free(), A.free()
    return out


def run_single(ctx, name, method, warmup, steps):
    sess = host.BenchSession(ctx, name, method, "none")
    info = sess.prepare(warmup)
    r = sess.run(steps)
    hist = sess.history(warmup + steps + 1)
    sess.close()
    return info, r["device_ms"] / steps, hist


def run_case(ctx, size, method, warmup, steps):
    name = f"HPCG-{size}"
    res = {"matrix": name, "method": method, "rounds": [], "block": []}
    per_k = {k: [] for k in KS}
    singles = []
    ok = True
    for rnd in range(2):
        info, single_ms, single_hist = run_single(ctx, name, method, warmup, steps)
        singles.append(single_ms)
        res.update({"n": info["n_rows"], "nnz": info["nnz"]})
        row = {"round": rnd, "single_ms_per_iter": single_ms, "block": []}
        for k in KS:
            B = rhs(info["n_rows"], k, 1000 + k)
            got, ms, iters = host.bench_block(ctx, name, B, "none", warmup, steps, method=method)
            h0 = got.histories[0]
            m = min(8, h0.size, single_hist.size)
            err = float(np.max(np.abs(h0[:m] - single_hist[:m])) / single_hist[0])
            ok = ok and err <= 1e-10
            e = {"k": k, "ms_per_iter": ms / iters, "ms_per_iter_per_rhs": ms / iters / k, "timed_iters": iters,
                 "launches_per_iter": got.launches / got.iterations,
                 "gain_per_rhs_vs_single": single_ms / (ms / iters / k), "sanity_first_residuals_rel_err": err}
            per_k[k].append(e)
            row["block"].append(e)
            print(json.dumps({"matrix": name, "method": method, "round": rnd, **e}), flush=True)
        res["rounds"].append(row)
    res["single_ms_per_iter_median"] = float(np.median(singles))
    for k in KS:
        ms = float(np.median([e["ms_per_iter"] for e in per_k[k]]))
        res["block"].append({"k": k, "ms_per_iter_median": ms, "ms_per_iter_per_rhs_median": ms / k,
                             "gain_per_rhs_vs_single_median": res["single_ms_per_iter_median"] / (ms / k)})
    res["sanity_ok"] = ok
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--sizes", default="128,256")
    a = ap.parse_args()
    if a.warmup < 5 or a.steps < 50:
        ap.error("at least 5 warm-up and 50 timed iterations")
    os.makedirs(a.out, exist_ok=True)
    ctx = capi.Context(0)
    ctx.set_option("vector_cache", 0)
    out = {"header": gpu_header(), "warmup": a.warmup, "steps": a.steps, "cases": [], "sweep": []}
    for size in [int(s) for s in a.sizes.split(",")]:
        sw = sweep_per_level(ctx, size)
        out["sweep"].append({"matrix": f"HPCG-{size}", **sw})
        print(json.dumps({"sweep": f"HPCG-{size}", **sw}), flush=True)
        for method in ("gs", "sgs"):
            out["cases"].append(run_case(ctx, size, method, a.warmup, a.steps))
    ctx.close()
    out["header_after"] = gpu_header()
    ok = all(c["sanity_ok"] for c in out["cases"])
    out["sanity_ok"] = ok
    with open(os.path.join(a.out, "block_gs.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"header": out["header"], "sanity_ok": ok}))
    if not ok:
        sys.exit("sanity check failed: block column 0 differs from the single-RHS run")


if __name__ == "__main__":
    main()
