"""Block CG (several right-hand sides, one matrix) against the single-RHS CG, on one GPU.

    python tools/run_block_cg.py --out <dir> [--warmup 5] [--steps 50] [--no-512]

One process, one output directory, one JSON file (block_cg.json).  Per size (HPCG-256 at k = 1, 2, 4, 8, 16;
HPCG-512 at k = 1, 2, 4, 8 where it fits in device memory) it records:
  - block CG ms/iter and ms/iter per right-hand side (CUDA events over `steps` iterations after `warmup`,
    tolerance 0, distinct seeded right-hand sides; column 0 is b = 1, x0 = 0.1 -- the single-RHS run's system);
  - the single-RHS CG ms/iter on the same matrix in the same process (host.BenchSession, "cg", "none");
  - bis_spmm ms per launch and TB/s over its compulsory bytes 12 nnz + rp_bytes (n+1) + 16 n k, and the x-gather
    rate 8 k nnz / time (what the SpMM asks of L1/L2);
  - the bytes model per iteration and right-hand side next to the measured times.
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


def gpu_header():
    out = {"gpu": None, "power_limit_w": None}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out = {"gpu": q[0].strip(), "power_limit_w": float(q[1]), "sm_max_mhz": float(q[2])}
    except Exception as e:  # the numbers below are still device-timed; the header says what is missing
        out["header_error"] = repr(e)
    return out


def bytes_model(n, nnz, rp_bytes, k):
    """HBM bytes per iteration and right-hand side, precond none: the single-RHS CG streams the matrix through the
    windowed SpMV (10 B/nnz) and 12 vector passes; the block CG reads the CRS (12 B/nnz) once for k columns."""
    single = 10 * nnz + rp_bytes * (n + 1) + 12 * 8 * n
    block = (12 * nnz + rp_bytes * (n + 1)) / k + 12 * 8 * n
    return single, block


def rhs(n, k, seed):
    B = np.empty((n, k))
    B[:, 0] = 1.0
    rng = np.random.default_rng(seed)
    for j in range(1, k):
        B[:, j] = rng.uniform(-1.0, 1.0, n)
    return B


def time_spmm(ctx, A, n, k, reps=20):
    X, Y = ctx.alloc(n * k), ctx.alloc(n * k)
    ctx.call("bis_init_vector", X, 0.5, n * k)
    for _ in range(3):
        ctx.spmm(A, X, Y, k)
    ctx.sync()
    ctx.timer_start()
    for _ in range(reps):
        ctx.spmm(A, X, Y, k)
    ms = ctx.timer_stop() / reps
    ctx.free(X), ctx.free(Y)
    return ms


def run_size(ctx, size, ks, warmup, steps, host_mem):
    name = f"HPCG-{size}"
    res = {"matrix": name, "single": None, "block": []}
    # single-RHS CG, same matrix, same process
    sess = host.BenchSession(ctx, name, "cg", "none")
    info = sess.prepare(warmup)
    r = sess.run(steps)
    single_hist = sess.history(warmup + steps + 1)
    sess.close()
    n, nnz, rp_bytes = info["n_rows"], info["nnz"], info["rp_bytes"]
    res["single"] = {"ms_per_iter": r["device_ms"] / steps, "launches_per_iter": r["launches"] / steps}
    res.update({"n": n, "nnz": nnz, "rp_bytes": rp_bytes})
    A = ctx.generate_hpcg(size)
    spmv_x, spmv_y = ctx.alloc(n), ctx.alloc(n)
    ctx.call("bis_init_vector", spmv_x, 0.5, n)
    ctx.call("bis_spmv", A.h, spmv_x, spmv_y)
    ctx.sync()
    ctx.timer_start()
    for _ in range(20):
        ctx.call("bis_spmv", A.h, spmv_x, spmv_y)
    res["spmv_ms"] = ctx.timer_stop() / 20
    ctx.free(spmv_x), ctx.free(spmv_y)
    for k in ks:
        entry = {"k": k}
        if A is None:
            A = ctx.generate_hpcg(size)
        if 16 * n * k + (1 << 30) <= ctx.info()["free"]:
            ms_spmm = time_spmm(ctx, A, n, k)
            spmm_bytes = 12 * nnz + rp_bytes * (n + 1) + 16 * n * k
            entry["spmm_ms"] = ms_spmm
            entry["spmm_TBps"] = spmm_bytes / (ms_spmm * 1e-3) / 1e12
            entry["spmm_gather_TBps"] = 8 * k * nnz / (ms_spmm * 1e-3) / 1e12
        else:
            entry["spmm_skipped"] = "X and Y do not fit next to the matrix"
        A.free()   # the block solve generates its own copy
        A = None
        free = ctx.info()["free"]
        need = 12 * nnz + rp_bytes * (n + 1) + 11 * 8 * n * k + 8 * n + (1 << 30)
        host_need = 3 * 8 * n * k
        if need > free or (host_mem and host_need > host_mem // 2):
            entry["skipped"] = (f"needs {need / 1e9:.1f} GB device, {host_need / 1e9:.1f} GB host; "
                                f"free {free / 1e9:.1f} GB device, {host_mem / 1e9:.1f} GB host")
            res["block"].append(entry)
            print(json.dumps({"matrix": name, **entry}), flush=True)
            continue
        B = rhs(n, k, 1000 + k)
        got, ms, iters = host.bench_block(ctx, name, B, "none", warmup, steps)
        del B
        entry["ms_per_iter"] = ms / iters
        entry["ms_per_iter_per_rhs"] = ms / iters / k
        entry["timed_iters"] = iters
        entry["launches_per_iter"] = got.launches / got.iterations
        entry["speedup_per_rhs_vs_single"] = res["single"]["ms_per_iter"] / entry["ms_per_iter_per_rhs"]
        m_single, m_block = bytes_model(n, nnz, rp_bytes, k)
        entry["model_bytes_per_iter_per_rhs"] = {"single": m_single / n, "block": m_block / n, "unit": "bytes / n"}
        entry["model_speedup"] = m_single / m_block
        if "spmm_ms" in entry:
            # the SpMM's share of the bytes model: compulsory SpMM bytes at the measured time vs the whole model
            entry["spmm_ms_per_rhs"] = entry["spmm_ms"] / k
        # sanity: column 0 is the single-RHS run's system
        h0 = got.histories[0]
        m = min(8, h0.size, single_hist.size)
        err = float(np.max(np.abs(h0[:m] - single_hist[:m])) / single_hist[0])
        entry["sanity_first_residuals_rel_err"] = err
        entry["sanity_ok"] = bool(err <= 1e-10)
        res["block"].append(entry)
        print(json.dumps({"matrix": name, **entry}), flush=True)
    if A is not None:
        A.free()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--no-512", action="store_true", help="HPCG-256 only")
    a = ap.parse_args()
    if a.warmup < 5 or a.steps < 50:
        ap.error("at least 5 warm-up and 50 timed iterations")
    os.makedirs(a.out, exist_ok=True)
    try:
        host_mem = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES")
    except (ValueError, OSError):
        host_mem = 0
    ctx = capi.Context(0)
    ctx.set_option("vector_cache", 0)   # free bytes as bis_context_info reports them are what the next size can use
    out = {"header": gpu_header(), "warmup": a.warmup, "steps": a.steps, "sizes": []}
    out["sizes"].append(run_size(ctx, 256, [1, 2, 4, 8, 16], a.warmup, a.steps, host_mem))
    if not a.no_512:
        out["sizes"].append(run_size(ctx, 512, [1, 2, 4, 8], a.warmup, a.steps, host_mem))
    ctx.close()
    ok = all(e.get("sanity_ok", True) for s in out["sizes"] for e in s["block"])
    out["sanity_ok"] = ok
    with open(os.path.join(a.out, "block_cg.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"header": out["header"], "sanity_ok": ok}))
    if not ok:
        sys.exit("sanity check failed: block column 0 differs from the single-RHS run")


if __name__ == "__main__":
    main()
