#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: PCG time/iteration and SpMV HBM GB/s vs roofline on HPCG-512.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--grid 512] [--dump-outputs DIR]

A "step" is ONE iteration of the solver harness loop (solver_harness.hpp:17-50 of the
reference: iterate, residual-norm sample read back by the host, pointer exchange) of
Jacobi-preconditioned CG (`-cg -p j`) on the HPCG-n 27-point matrix (default n = 512:
134 M rows, 3.6 G nonzeros, device-generated, 64-bit row_ptr), b = 1, x0 = 0.1.
For N > 1 (launched by torchrun, one rank per GPU) the rows are partitioned into N z-slabs
(strong scaling: the global problem is fixed; `--weak` keeps an HPCG-n slab per GPU instead); halo planes and
dot-product sums move over peer memory from inside the kernels (NCCL sets the link up and is the fallback).  `value` is milliseconds per iteration with all state resident in HBM (CUDA events,
max over ranks); `e2e` is the same metric through the host stack from HOST buffers (b, x0 uploaded,
x_star downloaded, residual norm read back every iteration); `roofline` is the SpMV kernel
(the dominant kernel) against the measured HBM peak; `cpu_baseline` is the unmodified reference
(oracle/_ref) timed on the host cores on a bounded sample.

`--impl reference` times the reference's own CPU implementation of the same path (rank 0 only).

`--dump-outputs DIR` (one GPU) writes what the timed loop computed in its last step, for comparing two builds output
for output (the inputs are the same on every run): DIR/residual_norms.npy, ||r_0|| .. ||r_(W+K)|| of the session, and
the iterate x_(W+K) at a fixed seeded sample of DUMP_X_SAMPLE rows, DIR/x_sample.npy (values) and
DIR/x_sample_rows.npy (row numbers); float64, 16 MB in all.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "pcg_time_per_iteration_hpcg"
UNIT = "ms/iter"


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks line),
    through NVML in a thread (1 ms period: the 8-GPU timed region is only tens of milliseconds long);
    nvidia-smi -lms as the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines: list[str] = []
        self.nvml = None
        self.sm: list[float] = []
        self.mask = 0
        self.mx = None
        self._stop = threading.Event()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = self.idx
            if vis:
                ids = [v for v in vis.split(",") if v.strip() != ""]
                if self.idx < len(ids) and ids[self.idx].strip().isdigit():
                    phys = int(ids[self.idx])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _poll(self):
        nv = self.nvml
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                pass
            time.sleep(0.001)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.nvml:
            self._stop.set()
            self.t.join(timeout=2)
            reasons = sorted(k for k, b in self.BITS.items() if self.mask & b)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.mx,
                    "samples": len(self.sm), "reasons": reasons, "source": "nvml, 1 ms period"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 100"}


def slab_rows(n: int, nz_planes: int, plane: int, rank: int, nranks: int):
    """Row block of `rank`: the library's own rule (bis_partition_row_block: unions of 8 fixed virtual
    slabs when nranks divides 8, which makes the reductions partition-invariant)."""
    from basic_iterative_solvers_b200 import capi
    return capi.partition_row_block(n, plane, rank, nranks)


# ---------------------------------------------------------------------------------------------
def reference_leg(n_sample: int, iters: int, threads: int | None, n_target: int):
    """The UNMODIFIED reference (oracle/_ref/libbis_ref.so: /root/reference compiled behind an
    extern-C shim) running `-cg -p j` on HPCG-<n_sample> with all host threads, `iters`
    iterations.  The CRS comes from oracle/matgen.py (numpy): nothing of the product is imported or
    loaded on this path.  Returns the measured ms/iter, and that number scaled to HPCG-<n_target> by
    the row ratio (every kernel on the path is linear in the rows; the reference cannot hold HPCG-512:
    32-bit nnz, SURVEY F5)."""
    from oracle import matgen, refshim
    if not refshim.available():
        raise RuntimeError("oracle/_ref/libbis_ref.so is missing (built by __graft_entry__.build() where "
                           "/root/reference exists)")
    lib = refshim.load()
    cores = threads or os.cpu_count() or 1
    try:
        cores = min(cores, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    os.environ.setdefault("OMP_PROC_BIND", "close")
    lib.ref_omp_set_threads(int(cores))
    t0 = time.time()
    rp, col, val = matgen.hpcg(n_sample)
    t_gen = time.time() - t0
    lib.ref_set_max_iters(int(iters))
    t0 = time.time()
    r = refshim.solve(rp, col, val, "cg", "j")
    wall = time.time() - t0
    lib.ref_set_max_iters(0)
    its = max(r.iter_count, 1)
    ms_iter = 1e3 * r.iterate_time / its                 # the reference's own "iterate" stopwatch
    spmv_ms = 1e3 * r.spmv_time / its                    # its "SpMV time" timer / SpMV count
    scale = (n_target / n_sample) ** 3
    nnz = int(rp[-1])
    nrow = rp.size - 1
    spmv_bytes = 12 * nnz + 4 * (nrow + 1) + 16 * nrow
    return {
        "value": ms_iter * scale, "unit": UNIT, "cores": int(cores), "kind": "reference",
        "sample": (f"HPCG-{n_sample} -cg -p j, {its} iterations of the reference's solve() at {cores} OpenMP "
                   f"threads: {ms_iter:.2f} ms/iter measured (SpMV {spmv_ms:.2f} ms = "
                   f"{spmv_bytes / spmv_ms / 1e6:.1f} GB/s)"
                   + (f", x{scale:.0f} row ratio to HPCG-{n_target}" if scale != 1 else "")
                   + f"; {wall:.1f} s of CPU work incl. its preprocessing, {t_gen:.0f} s numpy matrix generation"),
        "extrapolated": scale != 1, "sample_config": f"HPCG-{n_sample} -cg -p j", "scale": scale,
        "measured_ms_per_iter": ms_iter, "spmv_ms": spmv_ms, "spmv_gbs": spmv_bytes / spmv_ms / 1e6,
    }


def pick_cpu_sample(n_target: int) -> int:
    try:
        avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
    except (ValueError, OSError):
        avail = 0
    n = 256 if avail > 48 << 30 else 128
    return min(n, n_target)


PARITY_GOLDEN = os.path.join(ROOT, "tests", "golden", "bench_parity.json")
PARITY_LEN = 25
DUMP_X_SAMPLE = 1 << 20


def parity_block(histories: dict, n: int, world: int, write_to: str | None):
    """First residual norms of the bench workload (CG + Jacobi and BiCGSTAB + Jacobi) against the committed
    one-GPU golden of the same workload (tests/golden/bench_parity.json, written by `--write-parity-golden` on one
    GPU).  Reductions are partition-invariant, so the expected max_rel at 2, 4 and 8 GPUs is exactly 0."""
    key = f"hpcg{n}"
    out = {"n_residuals": PARITY_LEN, "golden": "tests/golden/bench_parity.json", "workload": f"HPCG-{n} -cg/-bi -p j"}
    if write_to and world == 1:
        rec = {}
        try:
            with open(PARITY_GOLDEN) as f:
                rec = json.load(f)
        except (OSError, ValueError):
            pass
        rec[key] = {m: [float(v).hex() for v in h] for m, h in histories.items()}
        os.makedirs(os.path.dirname(os.path.abspath(write_to)), exist_ok=True)
        with open(write_to, "w") as f:
            json.dump(rec, f, indent=1)
        out["written"] = write_to
    try:
        with open(PARITY_GOLDEN) as f:
            gold = json.load(f).get(key)
    except (OSError, ValueError):
        gold = None
    if not gold:
        out["status"] = "no golden for this grid"
        return out
    worst, bit = 0.0, True
    for m, h in histories.items():
        g = [float.fromhex(v) for v in gold[m]]
        k = min(len(g), len(h))
        r0 = g[0]
        d = max(abs(a - b) for a, b in zip(h[:k], g[:k])) / r0
        out[f"{m}_max_rel"] = d
        out[f"{m}_bit_identical"] = all(float(a).hex() == float(b).hex() for a, b in zip(h[:k], g[:k]))
        worst = max(worst, d)
        bit = bit and out[f"{m}_bit_identical"]
    out["max_rel"] = worst
    out["bit_identical"] = bit
    return out


# ---------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--grid", dest="n", type=int, default=512, help="HPCG grid edge (BASELINE: 512)")
    ap.add_argument("--weak", action="store_true",
                    help="weak scaling: every GPU keeps an HPCG-<grid> sized slab (global grid n x n x n*N)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-full-solve", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=0, help="HPCG edge of the CPU sample (0: auto)")
    ap.add_argument("--write-parity-golden", default=None, metavar="PATH",
                    help="one GPU: write the parity golden (merged with the committed one) to PATH")
    ap.add_argument("--option", action="append", default=[], metavar="KEY=INT", help="bis_context_set_option")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="one GPU: write what the timed loop computed in its last step to DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.warmup < 3:
        args.warmup = 3
    # one solver session runs at most MAX_ITERS = 1000 iterations: the warm-up, the timed steps and the initial residual
    if args.warmup > 997:
        ap.error("--warmup must be at most 997")
    if args.steps < 1 or args.warmup + args.steps + 1 >= 1000:
        ap.error(f"--steps must be in [1, {998 - args.warmup}] with --warmup {args.warmup}")
    if args.dump_outputs and (world > 1 or args.impl != "ours"):
        ap.error("--dump-outputs needs one GPU and --impl ours")
    n = args.n
    nz = n * world if args.weak else n
    n_rows_g, nnz_g = n * n * nz, (3 * n - 2) ** 2 * (3 * nz - 2)
    scaling = "weak" if args.weak else "strong"
    gname = f"HPCG-{n}-{n}-{nz}" if args.weak else f"HPCG-{n}"
    workload = f"{gname} -cg -p j (27-point, {n_rows_g} rows, {nnz_g} nnz, fp64 CRS, b=1, x0=0.1)"
    config = {"workload": workload, "rows": n_rows_g, "nnz": nnz_g,
              "partition": f"{world} row block(s) = unions of 8 fixed z-slabs" if world > 1 else "single GPU",
              "l2": "inputs larger than L2 (no flush): CRS alone is %.1f GB per GPU" %
                    (12 * nnz_g / world / 1e9)}

    if args.impl == "reference":
        if rank != 0:
            return
        n_s = args.cpu_sample or pick_cpu_sample(n)
        leg = reference_leg(n_s, args.steps + args.warmup, None, n)   # warm-up iterations are inside the one bounded solve
        if leg["extrapolated"]:
            config["workload"] = (f"{workload} -- REFERENCE ARM: measured on {leg['sample_config']} "
                                  f"({leg['measured_ms_per_iter']:.2f} ms/iter) and scaled x{leg['scale']:.0f} by the row "
                                  f"ratio, because the reference cannot hold HPCG-{n} (32-bit nnz)")
        out = {"impl": "reference", "metric": METRIC, "value": leg["value"], "unit": UNIT, "n_gpus": args.gpus,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": leg["value"],
               "higher_is_better": False, "scaling": scaling, "vs_baseline": None, "dtype": "f64",
               "data": "synthetic", "config": config,
               "cpu_baseline": {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample", "extrapolated",
                                                    "sample_config", "scale", "measured_ms_per_iter")},
               "e2e": {"value": leg["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
               "spmv_gbs": leg["spmv_gbs"]}
        print(json.dumps(out), flush=True)
        return

    # NCCL prints "NCCL version ..." on stdout: everything but the ONE JSON line goes to stderr (the process's
    # file descriptor 1 is pointed at stderr for the run; the line is written to the saved descriptor at the end)
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    from basic_iterative_solvers_b200 import capi, host

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    nccl_id = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt = torch.frombuffer(bytearray(capi.Context.nccl_unique_id()), dtype=torch.uint8).cuda()
        dist.broadcast(idt, 0)
        nccl_id = bytes(idt.cpu().numpy().tobytes())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ctx = capi.Context(local_rank, rank, world, nccl_id)
    for kv in args.option:
        k, v = kv.split("=")
        ctx.set_option(k, int(v))
    if world > 1:
        config["partition"] += (", halo planes and the 8 slab sums of every dot product over peer memory (NVLink stores "
                                "from inside the SpMV / reducing kernels, CUDA IPC)" if ctx.info()["peer_memory"]
                                else ", NCCL halo send/recv + allreduce")
    K, W = args.steps, args.warmup
    name = gname
    r_lo, r_hi = slab_rows(n_rows_g, nz, n * n, rank, world)
    n_local = r_hi - r_lo

    # ---- e2e: host buffers in, host buffer out (pinned), through the host stack -----------------
    b_h = torch.full((n_local,), 1.0, dtype=torch.float64).pin_memory()
    x0_h = torch.full((n_local,), 0.1, dtype=torch.float64).pin_memory()
    xs_h = torch.empty(n_local, dtype=torch.float64).pin_memory()
    sess = host.BenchSession(ctx, name, "cg", "j")
    sess.e2e(W, b_h.data_ptr(), x0_h.data_ptr(), xs_h.data_ptr())          # warm-up pass (allocators, NCCL)
    barrier()
    e = sess.e2e(K, b_h.data_ptr(), x0_h.data_ptr(), xs_h.data_ptr())
    barrier()
    e2e_ms = max_over_ranks(e["wall_ms"]) / K
    setup_ms = max_over_ranks(sess.setup_ms())
    assert e["iters"] == K and e["n_rows"] == n_local
    e2e_check = float(xs_h[:4].sum())
    # parity: the first residual norms of the bench workload against the committed one-GPU golden
    histories = {}
    ep = sess.e2e(PARITY_LEN - 1, b_h.data_ptr(), x0_h.data_ptr(), None)
    histories["cg_j"] = [float(v) for v in sess.history(PARITY_LEN)]
    # a REAL solve through the same path: TOL = 1e-14, MAX_ITERS = 1000, set-up included
    full = None
    if not args.no_full_solve:
        barrier()
        f = sess.e2e(0, b_h.data_ptr(), x0_h.data_ptr(), xs_h.data_ptr())
        barrier()
        full = {"iters": f["iters"], "wall_ms": max_over_ranks(f["wall_ms"]), "setup_ms": max_over_ranks(sess.setup_ms()),
                "final_true_residual_rel": f["res_true"] / f["res0"], "launches": f["launches"],
                "note": "solve() to TOL = 1e-14 or MAX_ITERS = 1000 from host b / x0 to host x_star; setup_ms (matrix "
                        "generation + SpMV tile format) is reported beside it, not inside wall_ms"}
        full["ms_per_iter"] = full["wall_ms"] / max(full["iters"], 1)
    sess.close()
    sessb = host.BenchSession(ctx, name, "bi", "j")
    sessb.e2e(PARITY_LEN - 1, b_h.data_ptr(), x0_h.data_ptr(), None)
    histories["bi_j"] = [float(v) for v in sessb.history(PARITY_LEN)]
    sessb.close()
    parity = parity_block(histories, n, world, args.write_parity_golden) if (rank == 0 and not args.weak) else None

    # ---- resident: K timed iterations between CUDA events, per-launch profiling OFF ------------------
    sess = host.BenchSession(ctx, name, "cg", "j")
    info = sess.prepare(W)
    if world > 1:
        ctx.dist_wait_read(reset=True)
    clocks = ClockSampler(local_rank)
    clocks.start()      # BEFORE the barrier: NVML initialisation takes a rank-dependent 1 - 20 ms, and a rank that enters
    barrier()           # the timed loop late makes every other rank wait for it inside the first reduction
    t_clk = time.time()
    r = sess.run(K)
    barrier()
    if args.dump_outputs:
        # the iterate of the last timed step, copied on the device now (the loop runs on below) and read back later
        x_last = ctx.alloc(n_local)
        sess.copy_x(x_last)
        dump = {"residual_norms": sess.history(W + K + 1)}
    waits = ctx.dist_wait_read(reset=True) if world > 1 else None
    # a short timed region (tens of ms at 8 GPUs) gives the sampler nothing to see: keep the same
    # iteration loop running, untimed and unreported, until the sampler has watched ~0.6 s of it
    extra = 0
    while time.time() - t_clk < 0.6 and extra < 400 and W + 3 * K + extra + 2 < 1000:   # MAX_ITERS bounds a session
        sess.run(K)
        extra += K
    barrier()
    clk = clocks.stop()
    clk["window"] = f"the {K} timed iterations + {extra} further iterations of the same loop (untimed)"
    if args.dump_outputs:
        x = ctx.download(x_last, n_local)
        ctx.free(x_last)
        rows = np.arange(n_local)
        if n_local > DUMP_X_SAMPLE:
            rows = np.sort(np.random.default_rng(0).choice(n_local, DUMP_X_SAMPLE, replace=False))
        dump["x_sample"] = x[rows]
        dump["x_sample_rows"] = rows.astype(np.float64)
        del x
        os.makedirs(args.dump_outputs, exist_ok=True)
        for fname, a in dump.items():
            np.save(os.path.join(args.dump_outputs, fname + ".npy"), a)
    dev_ms = max_over_ranks(r["device_ms"])
    launches = r["launches"]
    ms_iter = dev_ms / K
    # ---- second pass of the same loop for the roofline: per-launch event pairs on, graph replay off ---
    sess.close()
    ctx.set_option("graph", 0)
    sess = host.BenchSession(ctx, name, "cg", "j")
    sess.prepare(W)
    ctx.profile_enable(True)
    barrier()
    rp_ = sess.run(K)
    barrier()
    spmv_ms_total, spmv_cnt = ctx.profile_read("spmv")
    vec_ms_total, vec_cnt = ctx.profile_read("vector")
    ctx.profile_enable(False)
    ctx.set_option("graph", 1)
    prof_dev_ms = rp_["device_ms"]
    sess.close()
    spmv_ms = spmv_ms_total / max(spmv_cnt, 1)
    # bytes the kernel itself has to move per launch: 8 B value + 2 B local column id per nonzero, row_ptr,
    # x once, y once, and the dot operand (p) once; the CRS-equivalent figure (12 B / nnz, SURVEY 8(d)) beside it
    own_bytes = 10 * info["nnz"] + info["rp_bytes"] * (info["n_rows"] + 1) + 24 * info["n_rows"]
    crs_bytes = 12 * info["nnz"] + info["rp_bytes"] * (info["n_rows"] + 1) + 16 * info["n_rows"]
    achieved = own_bytes / spmv_ms / 1e6            # GB/s, this rank's SpMV (per GPU)
    peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak = float(json.load(f)["hbm_gbs"])
            peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy)"
    except (OSError, KeyError, ValueError):
        pass
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "spmv_traffic.json")) as f:
            t = json.load(f)
            if t.get("workload_n") == n and world == 1:
                traffic = t["dram_bytes_per_launch"]
                traffic_src = "static: " + t.get("source", "ncu --set full capture under profiles/")
    except (OSError, KeyError, ValueError):
        pass

    # ---- BiCGSTAB + Jacobi on the same matrix (BASELINE configs[4]) ---------------------------
    sess = host.BenchSession(ctx, name, "bi", "j")
    sess.prepare(W)
    barrier()
    rb = sess.run(K)
    barrier()
    bi_ms = max_over_ranks(rb["device_ms"]) / K
    sess.close()

    # ---- the timed workload once more with the lossless value dictionary (option spmv_vdict, off by default) ------
    vdict = None
    if world == 1 and rank == 0 and not args.weak:
        ctx.set_option("spmv_vdict", 1)
        try:
            sv = host.BenchSession(ctx, name, "cg", "j")
            sv.prepare(W)
            rv = sv.run(K)
            hv = [float(v) for v in sv.history(min(PARITY_LEN, W + K + 1))]
            sv.close()
            ctx.set_option("graph", 0)
            sv = host.BenchSession(ctx, name, "cg", "j")
            iv = sv.prepare(W)
            ctx.profile_enable(True)
            sv.run(K)
            v_ms, v_cnt = ctx.profile_read("spmv")
            ctx.profile_enable(False)
            vbytes = ctx.get_option("spmv_value_bytes")
            sv.close()
            v_own = (2 + vbytes) * iv["nnz"] + iv["rp_bytes"] * (iv["n_rows"] + 1) + 24 * iv["n_rows"]
            vdict = {"option": "spmv_vdict = 1 (a 1-byte index per nonzero into the <= 256 distinct values of the matrix instead of "
                               "the 8-byte value; same bits)",
                     "ms_per_iter": rv["device_ms"] / K, "spmv_ms_per_launch": v_ms / max(v_cnt, 1),
                     "value_bytes_per_nnz": vbytes, "own_bytes_per_launch": v_own,
                     "own_gbs": v_own / (v_ms / max(v_cnt, 1)) / 1e6,
                     "history_equals_value_streaming_run": hv == histories["cg_j"][:len(hv)],
                     "note": "not the headline: with 15 instead of 40 GB per launch the kernel is no longer HBM-bound (it is bound "
                             "by the rate of its bulk-copy requests), so it is reported beside the roofline line, not in it"}
        finally:
            ctx.set_option("graph", 1)
            ctx.set_option("spmv_vdict", 0)

    # ---- the same metric on the configuration the CPU reference can actually hold (one GPU) --------
    same = None
    if world == 1 and rank == 0 and not args.weak and n > 256:
        s2 = host.BenchSession(ctx, "HPCG-256", "cg", "j")
        n2 = 256 ** 3
        b2 = torch.full((n2,), 1.0, dtype=torch.float64).pin_memory()
        x2 = torch.full((n2,), 0.1, dtype=torch.float64).pin_memory()
        o2 = torch.empty(n2, dtype=torch.float64).pin_memory()
        s2.e2e(W, b2.data_ptr(), x2.data_ptr(), o2.data_ptr())
        e2 = s2.e2e(K, b2.data_ptr(), x2.data_ptr(), o2.data_ptr())
        s2.close()
        s2 = host.BenchSession(ctx, "HPCG-256", "cg", "j")
        s2.prepare(W)
        r2 = s2.run(K)
        h2 = s2.history(W + K + 1)
        s2.close()
        same = {"workload": "HPCG-256 -cg -p j", "gpu_ms_per_iter": r2["device_ms"] / K,
                "gpu_e2e_ms_per_iter": e2["wall_ms"] / K}
        # the residual norms of those W + K iterations against the UNMODIFIED reference's (committed fixture made by
        # tests/golden/make_golden_large.py from the compiled reference at 1 and at 8 OpenMP threads)
        gpath = os.path.join(ROOT, "tests", "golden", "large_hpcg256_cg_j.npz")
        if os.path.exists(gpath):
            g = np.load(gpath)
            k = min(h2.size, g["history"].size, g["history8"].size)
            r0 = float(g["history"][0])
            same["parity_vs_reference"] = {
                "golden": "tests/golden/large_hpcg256_cg_j.npz (reference, 1 OpenMP thread)",
                "n_residuals": int(k),
                "max_abs_diff_over_r0": float(np.max(np.abs(h2[:k] - g["history"][:k])) / r0),
                "max_abs_diff_vs_8_thread_run_over_r0": float(np.max(np.abs(h2[:k] - g["history8"][:k])) / r0),
                "reference_1_vs_8_threads_over_r0": float(np.max(np.abs(g["history8"][:k] - g["history"][:k])) / r0),
                "tolerance": "1e-10 * ||r0|| where the reference reproduces itself to that level (north_star); its own "
                             "1-thread and 8-thread runs are reported beside the device's distance for scale",
            }

    # ---- the triangular-solve configuration of BASELINE (configs[2]: HPCG-256 -cg -p sgs), one GPU ------------------
    sgs = None
    if world == 1 and rank == 0 and not args.weak and n > 256:
        ctx.set_option("graph", 0)      # per-launch event pairs need the launches issued one by one
        s3 = host.BenchSession(ctx, "HPCG-256", "cg", "sgs")
        s3.prepare(W)
        ctx.profile_enable(True)
        s3.run(K)
        trsv_ms, trsv_cnt = ctx.profile_read("sptrsv")
        ctx.profile_enable(False)
        ctx.set_option("graph", 1)
        s3.close()
        s3 = host.BenchSession(ctx, "HPCG-256", "cg", "sgs")
        s3.prepare(W)
        r3 = s3.run(K)
        h3 = s3.history(W + K + 1)
        s3.close()
        nnz_tri = (449455096 - 256 ** 3) // 2
        sweep_bytes = 12 * nnz_tri + 4 * (256 ** 3 + 1) + 24 * 256 ** 3     # SURVEY section 8(d)
        sgs = {"workload": "HPCG-256 -cg -p sgs (BASELINE configs[2])", "gpu_ms_per_iter": r3["device_ms"] / K,
               "sptrsv_ms_per_sweep": trsv_ms / trsv_cnt if trsv_cnt else None, "sweeps_timed": int(trsv_cnt),
               "sptrsv_kernel": "wave_kernel (stencil wavefront, thread-block clusters of 8 planes)",
               "sptrsv_algorithmic_gbs": sweep_bytes / (trsv_ms / trsv_cnt) / 1e6 if trsv_cnt else None,
               "note": "the sweeps are a dependency chain of 7n-6 levels: latency-bound by nature, rated in ms per sweep"}
        gpath = os.path.join(ROOT, "tests", "golden", "large_hpcg256_cg_sgs.npz")
        if os.path.exists(gpath):
            g = np.load(gpath)
            k = min(h3.size, g["history"].size, g["history8"].size)
            r0 = float(g["history"][0])
            sgs["parity_vs_reference"] = {
                "golden": "tests/golden/large_hpcg256_cg_sgs.npz (reference, 1 and 8 OpenMP threads)", "n_residuals": int(k),
                "max_abs_diff_over_r0": float(np.max(np.abs(h3[:k] - g["history"][:k])) / r0),
                "reference_1_vs_8_threads_over_r0": float(np.max(np.abs(g["history8"][:k] - g["history"][:k])) / r0)}

    out = {
        "metric": METRIC, "value": ms_iter, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_iter, "higher_is_better": False, "scaling": scaling, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config,
        "e2e": {"value": e2e_ms, "unit": UNIT,
                "h2d_bytes_per_step": 16 * n_local / K, "d2h_bytes_per_step": 8 * n_local / K + 8,
                "note": "preprocessing (allocate, upload b/x0 from pinned host memory, r0) + K harness "
                        "iterations with the residual norm read back each + x_star download, / K; the matrix set-up "
                        "(setup_ms: generation + SpMV tile format + order table, once per matrix) is outside",
                "setup_ms": setup_ms, "x_star_check": e2e_check, "breakdown_ms_rank0": e["breakdown_ms"],
                "full_solve": full},
        "gpu_launches": launches,
        "timing": "value: CUDA events around the K iterations, per-launch profiling OFF, iteration bodies replayed as "
                  "CUDA graphs on one GPU; roofline: a second pass of the same loop with per-launch event pairs",
        "clocks": clk,
        "roofline": {"bound": "hbm", "kernel": "spmv_win_kernel<long, EpiDot> (y = A p fused with (y,p); val, 16-bit local column ids, row_ptr slice and x windows by TMA)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": own_bytes,
                     "bytes_note": "the kernel's own compulsory bytes: 10 B per nonzero (value + 16-bit local column id), "
                                   "row_ptr, x once, y once, the dot operand once",
                     "crs_equivalent_bytes_per_launch": crs_bytes, "crs_equivalent_gbs": crs_bytes / spmv_ms / 1e6,
                     "ms_per_launch": spmv_ms, "launches_timed": spmv_cnt,
                     "share_of_step": spmv_ms_total / prof_dev_ms,
                     "frac_of_nominal_8tbs": achieved / 8000.0},
        "spmv_gbs": achieved,
        "vector_kernels_ms_per_iter": vec_ms_total / K,
        "residual_after_timed_steps": r["res_last"] / r["res0"],
        "parity": parity,
        "also": {"bicgstab_jacobi_ms_per_iter": bi_ms, "bicgstab_launches": rb["launches"]},
    }
    if waits is not None:
        out["dist_wait"] = {"rank": rank,
                            "reduction_wait_ms_per_iter": max_over_ranks(waits[0] / 1e6 / K),
                            "reductions": int(waits[1]),
                            "halo_wait_ms_per_iter": max_over_ranks(waits[2] / 1e6 / K),
                            "note": "globaltimer inside the kernels: how long the finalising block of a reduction waited for "
                                    "the other ranks' slab sums, and CTA 0's producer for the halo flags (max over ranks)"}
    if same is not None:
        out["same_config"] = same
    if sgs is not None:
        out["also"]["hpcg256_cg_sgs"] = sgs
    if vdict is not None:
        out["also"]["value_dictionary"] = vdict
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        try:
            n_s = args.cpu_sample or pick_cpu_sample(n)
            leg = reference_leg(n_s, 30, None, n)
            out["cpu_baseline"] = {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample", "extrapolated",
                                                       "sample_config", "scale", "measured_ms_per_iter")}
            if same is not None and n_s == 256:
                same["cpu_ms_per_iter"] = leg["measured_ms_per_iter"]
                same["ratio"] = leg["measured_ms_per_iter"] / same["gpu_ms_per_iter"]
                same["e2e_ratio"] = leg["measured_ms_per_iter"] / same["gpu_e2e_ms_per_iter"]
        except Exception as ex:  # the baseline is a reported number, never a reason to lose the GPU line
            out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference",
                                   "sample": f"unavailable: {ex}"}
    ctx.close()
    if rank == 0:
        os.write(json_fd, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
