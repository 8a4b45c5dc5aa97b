"""Per-role cycle counters of the windowed SpMV (bis_spmv_win.cuh: WinStamp) on device-generated HPCG-n, dot-fused
launch as CG calls it.  Needs a library built with -DBIS_PERF_DEBUG, e.g.
   make -C basic_iterative_solvers_b200/csrc OUTDIR=/tmp/bisdbg EXTRA=-DBIS_PERF_DEBUG
   python tools/run_spmv_stamps.py /tmp/bisdbg/libbis_b200.so 512 [key=value ...]
Prints, per tile, the cycles each role spends in each phase (producer: lane 0 of its warp; consumers: mean over warps)."""
import os
import sys
import tempfile

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from basic_iterative_solvers_b200 import capi  # noqa: E402

capi.LIB_PATH = os.path.abspath(sys.argv[1])
n = int(sys.argv[2])
NAMES = ["p_empty_wait", "p_fence_expect_issue", "p_tiles", "p_total", "c_order_wait", "c_full_wait",
         "c_epilogue_load_wait", "c_walk_epilogue", "c_tiles", "c_total"]
with tempfile.TemporaryDirectory() as tmp, capi.Context(0) as ctx:
    path = os.path.join(tmp, "stamps.bin")
    os.environ["BIS_SPMV_STAMPS"] = path
    for kv in sys.argv[3:]:
        k, v = kv.split("=")
        ctx.set_option(k, int(v))
    A = ctx.generate_hpcg(n)
    N = A.info()["n_rows"]
    x, y = ctx.alloc(N), ctx.alloc(N)
    ctx.call("bis_init_vector", x, 1.0, N)

    def launch():
        ctx.call("bis_spmv_dot", A.h, x, y, x, 40, -1)

    for dbg in (0, 4):
        ctx.set_option("spmv_debug", dbg)
        launch()
        ctx.sync()
        ctx.timer_start()
        for _ in range(5):
            launch()
        ms = ctx.timer_stop() / 5
        print(f"HPCG-{n} {sys.argv[3:]} spmv_debug={dbg}: {ms:.3f} ms per launch, "
              f"{ctx.get_option('spmv_value_bytes')} B values, {ctx.get_option('spmv_stream_mb') / 1e3:.2f} GB compulsory")
    ctx.set_option("spmv_debug", 0)
    raw = np.fromfile(path, dtype=np.uint64).reshape(-1, 16)[-1].astype(np.float64)
    s = dict(zip(NAMES, raw[:10]))
    grid = int(raw[15])
    pt, ct = s["p_tiles"], s["c_tiles"]
    warps = ct / pt   # consumer warps per tile
    print(f"grid {grid} CTAs, {int(pt)} tiles, {warps:.0f} consumer warps per tile")
    print("producer per tile (cycles): " + ", ".join(f"{k[2:]} {s[k] / pt:.0f}" for k in
                                                       ("p_empty_wait", "p_fence_expect_issue")) +
          f", rest of the loop {(s['p_total'] - s['p_empty_wait'] - s['p_fence_expect_issue']) / pt:.0f}; "
          f"loop per tile and CTA {s['p_total'] / pt:.0f}")
    print("consumer warp per tile (cycles): " + ", ".join(f"{k[2:]} {s[k] / ct:.0f}" for k in
                                                         ("c_order_wait", "c_full_wait", "c_epilogue_load_wait",
                                                          "c_walk_epilogue")) +
          f"; loop per tile of the warp's group {s['c_total'] / ct:.0f}")
