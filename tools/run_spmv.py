"""Run a few plain SpMV launches on device-generated HPCG-n (profiling target):
   python tools/run_spmv.py n reps [key=value ...]   e.g. spmv_rows=256 spmv_stages=2"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from basic_iterative_solvers_b200 import capi  # noqa: E402

n, reps = int(sys.argv[1]), int(sys.argv[2])
with capi.Context(0) as ctx:
    kind = "spmv"
    for kv in sys.argv[3:]:
        k, v = kv.split("=")
        if k == "kind":
            kind = v
        else:
            ctx.set_option(k, int(v))
    A = ctx.generate_hpcg(n)
    inf = A.info()
    x, y = ctx.alloc(inf["n_rows"]), ctx.alloc(inf["n_rows"])
    ctx.call("bis_init_vector", x, 1.0, inf["n_rows"])
    def launch():
        if kind == "dot":
            ctx.call("bis_spmv_dot", A.h, x, y, x, 40, -1)
        else:
            ctx.call("bis_spmv", A.h, x, y)

    launch()   # builds the tile format (variant 3) on first use
    ctx.sync()
    ctx.timer_start()
    for _ in range(reps):
        launch()
    ms = ctx.timer_stop() / reps
    # the windowed kernel's own compulsory bytes, from its format's byte model (C library, option spmv_stream_mb)
    own = ctx.get_option("spmv_stream_mb") * 1e6
    print(f"HPCG-{n} {sys.argv[3:]}: {ms:.3f} ms  {A.spmv_bytes()/ms/1e6:.1f} GB/s CRS-equivalent  "
          f"own {own/1e9:.2f} GB/launch ({ctx.get_option('spmv_value_bytes')} B values) {own/ms/1e6:.1f} GB/s")
