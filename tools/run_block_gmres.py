"""Block GMRES (several right-hand sides, one matrix) against the single-RHS GMRES, on one GPU.

    python tools/run_block_gmres.py --out <dir> [--warmup 10] [--steps 50] [--rounds 2] [--small]

One process, one output directory, one JSON file (block_gmres.json).  Configurations (restart length 10):
Anderson 100x100x50 (ranpot 5) with Jacobi, and HPCG-256 without a preconditioner (--small: Anderson 40x40x20 and
HPCG-64, a rehearsal), at k = 1, 2, 4, 8, 16 where device and host memory allow.  Per configuration and k:
  - block GMRES ms/iter and ms/iter per right-hand side (CUDA events over the iterations after `warmup`, tolerance 0;
    column 0 is b = 1, x0 = INIT_X_VAL -- the single-RHS run's system, the others seeded uniform(-1, 1));
  - the single-RHS GMRES ms/iter on the same matrix in the same process (host.BenchSession "gm"), the two measured
    alternately `rounds` times after a warm-up; the lowest of each is reported next to every round's value;
  - the host time of the per-column Givens updates (least_squares + update_g), host clock, per loop iteration;
  - the bytes model per iteration and right-hand side (iteration body only, restarts excluded) and its gain.
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

M = 10
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


def bytes_model(n, nnz, rp_bytes, k, jacobi, spmv_stream_bytes):
    """HBM bytes per iteration and right-hand side, averaged over the basis indices i = 0..M-1 of a cycle (restarts
    excluded).  Vectors, 8 B per element and pass, the same per column in both: SpMV x, y (2); Jacobi w, D, w (3);
    h_0 (2); MGS step l < i: w, v_l, v_l+1, w (4), step i: w, v_i, w (3); scale w, v (2).  Matrix: the single-RHS
    GMRES streams it through the windowed SpMV (its own byte model as the library reports it, x and y included);
    the block reads the CRS (12 B/nnz + row pointers) once for its k columns."""
    vec = np.mean([2 + (3 if jacobi else 0) + 2 + 4 * i + 3 + 2 for i in range(M)]) * 8 * n
    single = spmv_stream_bytes + vec - 16 * n
    block = (12 * nnz + rp_bytes * (n + 1)) / k + vec
    return single, block


def rhs(n, k, seed):
    B = np.empty((n, k))
    B[:, 0] = 1.0
    rng = np.random.default_rng(seed)
    for j in range(1, k):
        B[:, j] = rng.uniform(-1.0, 1.0, n)
    return B


def single_run(ctx, name, precond, warmup, steps):
    sess = host.BenchSession(ctx, name, "gm", precond, restart_len=M)
    try:
        info = sess.prepare(warmup)
        r = sess.run(steps)
        hist = sess.history(warmup + steps + 1)
    finally:
        sess.close()
    return info, r["device_ms"] / steps, r["launches"] / steps, hist


def run_config(ctx, name, precond, warmup, steps, rounds, host_mem):
    res = {"matrix": name, "precond": precond, "restart_len": M, "single": {}, "block": []}
    info, _, _, single_hist = single_run(ctx, name, precond, warmup, steps)   # warm-up of the single-RHS path
    n, nnz, rp_bytes = info["n_rows"], info["nnz"], info["rp_bytes"]
    stream = ctx.get_option("spmv_stream_mb") * 1e6   # the session's last SpMV (windowed: its compulsory bytes)
    if stream == 0:
        stream = 12 * nnz + rp_bytes * (n + 1) + 16 * n
    res.update({"n": n, "nnz": nnz, "rp_bytes": rp_bytes, "single_spmv_stream_bytes": stream})
    singles = []
    for k in KS:
        entry = {"k": k}
        free = ctx.info()["free"]
        need = 12 * nnz + rp_bytes * (n + 1) + 8 * n * k * (M + 1 + 5) + 8 * n + (1 << 30)
        host_need = 3 * 8 * n * k
        if need > free or (host_mem and host_need > host_mem // 2):
            entry["skipped"] = (f"needs {need / 1e9:.1f} GB device, {host_need / 1e9:.1f} GB host; "
                                f"free {free / 1e9:.1f} GB device, {host_mem / 1e9:.1f} GB host")
            res["block"].append(entry)
            print(json.dumps({"matrix": name, **entry}), flush=True)
            continue
        B = rhs(n, k, 1000 + k)
        host.bench_block(ctx, name, B, precond, 5, 5, method="gm", restart_len=M)   # warm-up of this shape
        block_ms, single_ms, givens = [], [], []
        got = iters = None
        for _ in range(rounds):   # alternate: single, block
            _, s_ms, s_launch, _ = single_run(ctx, name, precond, warmup, steps)
            single_ms.append(s_ms)
            singles.append(s_ms)
            st = {}
            got, ms, iters = host.bench_block(ctx, name, B, precond, warmup, steps, method="gm", restart_len=M, stats=st)
            block_ms.append(ms / iters)
            givens.append(st["host_givens_s"] * 1e3 / got.iterations)
            res["single"]["launches_per_iter"] = s_launch
        del B
        best = min(block_ms)
        entry["ms_per_iter"] = best
        entry["ms_per_iter_rounds"] = block_ms
        entry["ms_per_iter_per_rhs"] = best / k
        entry["single_ms_per_iter"] = min(single_ms)
        entry["single_ms_per_iter_rounds"] = single_ms
        entry["speedup_per_rhs_vs_single"] = min(single_ms) / (best / k)
        entry["timed_iters"] = iters
        entry["launches_per_iter"] = got.launches / got.iterations
        entry["host_givens_ms_per_iter"] = min(givens)
        entry["host_givens_ms_per_iter_rounds"] = givens
        m_single, m_block = bytes_model(n, nnz, rp_bytes, k, precond == "j", stream)
        entry["model_bytes_per_iter_per_rhs"] = {"single": m_single, "block": m_block}
        entry["model_speedup"] = m_single / m_block
        h0 = got.histories[0]
        mm = min(8, h0.size, single_hist.size)
        err = float(np.max(np.abs(h0[:mm] - single_hist[:mm])) / single_hist[0])
        entry["sanity_first_residuals_rel_err"] = err
        entry["sanity_ok"] = bool(err <= 1e-10)
        res["block"].append(entry)
        print(json.dumps({"matrix": name, **entry}), flush=True)
    res["single"]["ms_per_iter"] = min(singles) if singles else None
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--small", action="store_true", help="rehearsal sizes: Anderson 40x40x20, HPCG-64")
    a = ap.parse_args()
    if a.warmup < 5 or a.steps < 20 or a.rounds < 1:
        ap.error("at least 5 warm-up and 20 timed iterations, and one round")
    if a.warmup + a.steps >= host.MAX_ITERS:
        ap.error("warmup + steps must stay below MAX_ITERS")
    os.makedirs(a.out, exist_ok=True)
    try:
        host_mem = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES")
    except (ValueError, OSError):
        host_mem = 0
    configs = ([("Anderson,Lx=40,Ly=40,Lz=20,ranpot=5.0,t=1.0,seed=1", "j"), ("HPCG-64", "none")] if a.small else
               [("Anderson,Lx=100,Ly=100,Lz=50,ranpot=5.0,t=1.0,seed=1", "j"), ("HPCG-256", "none")])
    ctx = capi.Context(0)
    ctx.set_option("vector_cache", 0)   # free bytes as bis_context_info reports them are what the next k can use
    out = {"header": gpu_header(), "warmup": a.warmup, "steps": a.steps, "rounds": a.rounds, "configs": []}
    for name, precond in configs:
        out["configs"].append(run_config(ctx, name, precond, a.warmup, a.steps, a.rounds, host_mem))
    ctx.close()
    ok = all(e.get("sanity_ok", True) for c in out["configs"] for e in c["block"])
    out["sanity_ok"] = ok
    with open(os.path.join(a.out, "block_gmres.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"header": out["header"], "sanity_ok": ok}))
    if not ok:
        sys.exit("sanity check failed: block column 0 differs from the single-RHS run")


if __name__ == "__main__":
    main()
