"""Kernels past 2^31 nonzeros and 2^31 block elements, checked against the slab-wise oracle (oracle/port.py).

HPCG-512 -- the benchmark's matrix, 3,609,741,304 nonzeros -- is where the library switches to 64-bit row_ptr and
where the offsets of the windowed SpMV (value-dictionary index, values), the SpMM tiles and the block streaming
kernels pass 2^31.  The whole-matrix oracle cannot hold such a matrix (int row_ptr), so the reference applies it
one row slab at a time, from templates (port.hpcg_slabs, port.anderson_slabs); tests/test_slab_oracle_cpu.py
shows that this has the bits of the whole-matrix oracle.

 a. HPCG-512: bis_spmv in every variant and every fused form, bit for bit; with integer-valued vectors every
    reduced scalar is an exact integer, so a dropped or doubled row shows in the slot whatever the reduction tree.
 b. Anderson 700 x 700 x 630 (more than 256 distinct values: the value-streaming windowed path), open and periodic.
 c. bis_spmm on HPCG 512 x 512 x 520 with k = 16: n*k = 2,181,038,080 elements.
 d. The block streaming kernels at the same n*k, on dyadic data where every operation is exact.
 e. bis_sptrsv / bis_bsptrsv / SGS on the HPCG-512 factors (1,737,761,788 nonzeros each, the dataflow solve).
 f. The 2^31 guard of bis_matrix_split_triangular (HPCG 512 x 512 x 640).
 g. Three CG + Jacobi iterations on HPCG-512 against a numpy restatement and tests/golden/bench_parity.json.

Each large matrix is built once by a class-scoped fixture and freed before the next one is built.  The device
memory each needs is computed from its size, not measured; the fixtures check that it is free.
"""
import contextlib
import json
import math
import os
import time
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import GOLDEN, HIST_TOL
from oracle import matgen, port

from basic_iterative_solvers_b200 import capi, host

pytestmark = pytest.mark.gpu

GB = 1e9
OPTIONS = ("spmv_variant", "spmv_vdict", "spmv_lanes", "factor_keep_crs")
PLANES = 4              # grid planes per oracle slab: about 1 M rows at 512 x 512, 2 M at 700 x 700
INT31 = 2 ** 31
RED_TOL = 1e-13         # the vector-CRS variant's rule (tests/test_kernels_gpu.py)
_PEAK = [0]


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def assert_bits(got, want, what):
    bad = np.flatnonzero(bits(got) != bits(want))
    assert bad.size == 0, (f"{what}: {bad.size} of {want.size} elements differ; first at {bad[:4].tolist()}: "
                           f"got {got[bad[:4]].tolist()}, want {want[bad[:4]].tolist()}")


def assert_exact(got, want, what):
    """a device scalar against an exact value (Python int or float that is exactly representable)"""
    w = np.float64(want)
    assert float(w) == want, f"{what}: {want} is not representable"
    assert bits(np.array([got]))[0] == bits(np.array([w]))[0], f"{what}: got {got!r}, want {want!r}"


def track(ctx):
    """peak device memory in use during the current test, sampled where the big buffers are live"""
    inf = ctx.info()
    _PEAK[0] = max(_PEAK[0], inf["total"] - inf["free"])


def release_vector_cache(ctx):
    """the context keeps freed vectors for reuse (option vector_cache, up to 48 GB): hand them back to the device"""
    on = ctx.get_option("vector_cache")
    ctx.set_option("vector_cache", 0)
    ctx.set_option("vector_cache", on)


def need(ctx, gbytes, what):
    release_vector_cache(ctx)
    free = ctx.info()["free"]
    assert free >= gbytes * GB, f"{what} needs about {gbytes} GB of free device memory, {free / GB:.1f} GB free"


@contextlib.contextmanager
def options(ctx, **kv):
    """set options for the duration of the block; every option of OPTIONS is restored afterwards"""
    saved = {k: ctx.get_option(k) for k in OPTIONS}
    try:
        for k, v in kv.items():
            ctx.set_option(k, v)
        yield
    finally:
        for k, v in saved.items():
            ctx.set_option(k, v)


@pytest.fixture(scope="module", autouse=True)
def _module_memory(ctx):
    """the module leaves no device memory allocated (torch, which holds the block tests' buffers, is set up first:
    its own context state is not an allocation of these tests)"""
    import torch
    torch.zeros(1, device="cuda")
    torch.cuda.synchronize()
    release_vector_cache(ctx)
    free0 = ctx.info()["free"]
    yield
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    release_vector_cache(ctx)
    free1 = ctx.info()["free"]
    print(f"\n[past-int32] device free before {free0 / GB:.3f} GB, after {free1 / GB:.3f} GB")
    assert free1 >= free0 - (256 << 20), f"the module left {(free0 - free1) / 2**20:.0f} MB allocated"


@pytest.fixture(autouse=True)
def _case(ctx, request):
    """runtime and peak device memory of each case; every option is restored afterwards"""
    _PEAK[0] = 0
    track(ctx)
    t0 = time.perf_counter()
    with options(ctx):
        yield
    print(f"\n[past-int32] {request.node.nodeid.split('::', 1)[1]}: {time.perf_counter() - t0:.1f} s, "
          f"peak device memory in use {_PEAK[0] / GB:.1f} GB")


def device_vectors(ctx, *arrays):
    return [ctx.upload(a) for a in arrays]


def spmv(ctx, A, dx, n):
    dy = ctx.alloc(n)
    try:
        ctx.call("bis_spmv", A.h, dx, dy)
        track(ctx)
        return ctx.download(dy, n)
    finally:
        ctx.free(dy)


# ---- a, e, g: HPCG-512 ---------------------------------------------------------------------------------------
@pytest.fixture(scope="class")
def hpcg512(ctx):
    n = 512 ** 3
    need(ctx, 60, "HPCG-512 (CRS 44 GB, window format and dictionary 11 GB)")
    t0 = time.perf_counter()
    with options(ctx, spmv_variant=0, spmv_vdict=1):
        A = ctx.generate_hpcg(512)
    t1 = time.perf_counter()
    slabs = port.hpcg_slabs(512, 512, 512, PLANES)
    x = np.random.default_rng(51).uniform(-1.0, 1.0, n)
    y = port.spmv_slabwise(slabs, x)
    print(f"\n[past-int32] HPCG-512: device generation {t1 - t0:.1f} s, oracle templates and one SpMV "
          f"{time.perf_counter() - t1:.1f} s")
    try:
        yield SimpleNamespace(A=A, n=n, slabs=slabs, x=x, y=y)
    finally:
        A.free()


class TestHpcg512:
    def test_info(self, ctx, hpcg512):
        inf = hpcg512.A.info()
        assert inf["n_rows"] == 134_217_728
        assert inf["nnz"] == 3_609_741_304 == matgen.hpcg_nnz(512)
        assert inf["rp_bytes"] == 8

    @pytest.mark.parametrize("config", ["auto_vdict", "windowed_no_vdict", "variant2", "variant1", "x_offset"])
    def test_spmv(self, ctx, hpcg512, config):
        A, n, x, y_ref = hpcg512.A, hpcg512.n, hpcg512.x, hpcg512.y
        opts = {"auto_vdict": dict(spmv_variant=0, spmv_vdict=1),
                "windowed_no_vdict": dict(spmv_variant=0, spmv_vdict=0),
                "variant2": dict(spmv_variant=2),
                "variant1": dict(spmv_variant=1),
                "x_offset": dict(spmv_variant=0, spmv_vdict=1)}[config]
        with options(ctx, **opts):
            if config == "x_offset":
                # x one double past a 16-byte boundary: the windowed kernel cannot take it, auto falls back to 2
                base = ctx.alloc(n + 1)
                dx = base + 8
            else:
                base = dx = ctx.alloc(n)
            try:
                ctx.upload(x, dx)
                y = spmv(ctx, A, dx, n)
                value_bytes = ctx.get_option("spmv_value_bytes")
            finally:
                ctx.free(base)
        if config == "variant1":
            err = np.max(np.abs(y - y_ref)) / np.max(np.abs(y_ref))
            assert err <= RED_TOL, err
        else:
            assert_bits(y, y_ref, config)
        if config == "auto_vdict":
            assert value_bytes == 1, "the windowed SpMV dropped the value dictionary"
        if config == "windowed_no_vdict":
            assert value_bytes == 8

    @pytest.mark.parametrize("vdict", [1, 0])
    def test_fused_forms(self, ctx, hpcg512, vdict):
        """every fused form against the oracle's y composed as the reference composes it"""
        A, n, x, y = hpcg512.A, hpcg512.n, hpcg512.x, hpcg512.y
        rng = np.random.default_rng(52)
        v, D = rng.uniform(-1.0, 1.0, n), rng.uniform(1.0, 2.0, n)
        with options(ctx, spmv_variant=0, spmv_vdict=vdict):
            out = fused_forms(ctx, A, x, v, D)
        assert_bits(out["dot_y"], y, "spmv_dot y")
        assert_bits(out["res_r"], v - y, "spmv_residual r")
        assert_bits(out["res_t"], y, "spmv_residual A x")
        jac = (v - (y - D * x)) / D
        assert_bits(out["jac"], jac, "spmv_jacobi")
        assert_bits(out["jacr_x"], jac, "spmv_jacobi_residual x")
        assert_bits(out["jacr_r"], v - y, "spmv_jacobi_residual r")
        r = v - y
        nrm = np.linalg.norm
        for got, a, b, what in ((out["dot_s"][0], y, v, "(y, w)"), (out["dot_s"][1], y, y, "(y, y)"),
                                (out["dotx_s"][0], y, x, "(y, x)"), (out["res_s"], r, r, "(r, r)"),
                                (out["jacr_s"], r, r, "jacobi (r, r)")):
            assert abs(got - a @ b) <= 1e-12 * nrm(a) * nrm(b), (what, got, a @ b)

    @pytest.mark.parametrize("vdict", [1, 0])
    def test_fused_scalars_exact_on_integers(self, ctx, hpcg512, vdict):
        """x, v integers in [-8, 8]: every product and partial sum is an exact integer below 2^53, so every slot
        equals the exact sum whatever the reduction tree -- a row dropped or counted twice changes it"""
        A, n, slabs = hpcg512.A, hpcg512.n, hpcg512.slabs
        rng = np.random.default_rng(53)
        xi, vi = rng.integers(-8, 9, n), rng.integers(-8, 9, n)
        x, v, D = xi.astype(np.float64), vi.astype(np.float64), np.full(n, 2.0)
        y = port.spmv_slabwise(slabs, x)
        yi = y.astype(np.int64)
        assert np.array_equal(yi.astype(np.float64), y)
        with options(ctx, spmv_variant=0, spmv_vdict=vdict):
            out = fused_forms(ctx, A, x, v, D)
        assert_bits(out["dot_y"], y, "spmv_dot y")
        assert_bits(out["res_r"], v - y, "spmv_residual r")
        assert_bits(out["jacr_r"], v - y, "spmv_jacobi_residual r")
        ri = vi - yi
        exact = {"(y, w)": (out["dot_s"][0], int(yi @ vi)), "(y, y)": (out["dot_s"][1], int(yi @ yi)),
                 "(y, x)": (out["dotx_s"][0], int(yi @ xi)), "(y, y) with w = x": (out["dotx_s"][1], int(yi @ yi)),
                 "(r, r)": (out["res_s"], int(ri @ ri)), "jacobi (r, r)": (out["jacr_s"], int(ri @ ri))}
        for what, (got, want) in exact.items():
            assert abs(want) < 2 ** 53
            assert_exact(got, want, what)

    def test_triangular_solves(self, ctx, hpcg512):
        """forward, backward and SGS on the strict factors, as the host builds them for -p sgs"""
        A, n, slabs = hpcg512.A, hpcg512.n, hpcg512.slabs
        need(ctx, 50, "the HPCG-512 factors")
        with options(ctx, factor_keep_crs=0):
            L, U = ctx.split_triangular(A)
        try:
            track(ctx)
            for T in (L, U):
                inf = T.info()
                assert inf["nnz"] == 1_737_761_788 and inf["rp_bytes"] == 4, inf
            dD, dDi = ctx.alloc(n), ctx.alloc(n)
            ctx.call("bis_matrix_extract_diagonal", A.h, dD, dDi)
            D = ctx.download(dD, n)
            assert np.all(D == 26.0)
            b = np.random.default_rng(54).uniform(-1.0, 1.0, n)
            fwd = port.sptrsv_slabwise(slabs, D, b)
            mid = (fwd * 1.0) * D
            bwd = port.sptrsv_slabwise(slabs, D, mid, backward=True)
            db, dmid = device_vectors(ctx, b, mid)
            dx, dtmp, dwork = ctx.alloc(n), ctx.alloc(n), ctx.alloc(n)
            track(ctx)
            ctx.call("bis_sptrsv", L.h, dx, dD, db)
            assert_bits(ctx.download(dx, n), fwd, "bis_sptrsv")
            ctx.call("bis_bsptrsv", U.h, dx, dD, dmid)
            assert_bits(ctx.download(dx, n), bwd, "bis_bsptrsv")
            ctx.call("bis_init_vector", dx, float("nan"), n)
            ctx.call("bis_apply_preconditioner", capi.PRECOND["sgs"], n, L.h, U.h, dD, dDi, dD, dD, dx, db, dtmp, dwork)
            assert_bits(ctx.download(dx, n), bwd, "SGS")
            print(f"\n[past-int32] factor levels: L {L.info()['n_levels']}, U {U.info()['n_levels']}")
            for d in (dD, dDi, db, dmid, dx, dtmp, dwork):
                ctx.free(d)
        finally:
            L.free()
            U.free()

    def test_cg_jacobi_residuals(self, ctx, hpcg512):
        """three CG + Jacobi iterations (b = 1, x0 = 0.1): numpy restatement of cg.hpp with A p from the slab
        oracle, the committed bench golden and the device solve agree within HIST_TOL * ||r0||"""
        n, slabs = hpcg512.n, hpcg512.slabs
        need(ctx, 60, "the device solve's own HPCG-512")
        D = np.full(n, 26.0)
        b, x = np.ones(n), np.full(n, 0.1)
        r = b - port.spmv_slabwise(slabs, x)
        z = r / D
        p = z.copy()
        hist = [math.sqrt(r @ r)]
        for _ in range(3):
            Ap = port.spmv_slabwise(slabs, p)
            rz = r @ z
            alpha = rz / (Ap @ p)
            x += alpha * p
            r -= alpha * Ap
            z = r / D
            beta = (r @ z) / rz
            p = z + beta * p
            hist.append(math.sqrt(r @ r))
        hist = np.array(hist)
        with open(os.path.join(GOLDEN, "bench_parity.json")) as f:
            gold = np.array([float.fromhex(v) for v in json.load(f)["hpcg512"]["cg_j"][:4]])
        got = host.solve(ctx, "cg", "j", matrix_name="HPCG-512", max_iters=3, want_x=False)
        track(ctx)
        dev = got.history[:4]
        assert dev.size == 4
        r0 = hist[0]
        for what, h in (("bench golden", gold), ("device solve", dev)):
            err = np.max(np.abs(h - hist)) / r0
            assert err <= HIST_TOL, (what, err, h, hist)


def fused_forms(ctx, A, x, v, D):
    """the fused forms of tests/test_spmv_vdict_default_gpu.py::_fused_forms that take the whole matrix"""
    n = x.size
    dx, dv, dD = device_vectors(ctx, x, v, D)
    dy, dr, dt, dxn = (ctx.alloc(n) for _ in range(4))
    track(ctx)
    out = {}
    try:
        ctx.call("bis_spmv_dot", A.h, dx, dy, dv, 20, 21)
        out["dot_y"], out["dot_s"] = ctx.download(dy, n), ctx.scalars(20, 2)
        ctx.call("bis_spmv_dot", A.h, dx, dy, dx, 22, 23)
        out["dotx_s"] = ctx.scalars(22, 2)
        ctx.call("bis_spmv_residual", A.h, dx, dv, dr, dt, 24)
        out["res_r"], out["res_t"], out["res_s"] = ctx.download(dr, n), ctx.download(dt, n), ctx.scalars(24)[0]
        ctx.call("bis_spmv_jacobi", A.h, dD, dv, dx, dxn)
        out["jac"] = ctx.download(dxn, n)
        ctx.call("bis_init_vector", dxn, float("nan"), n)
        ctx.call("bis_spmv_jacobi_residual", A.h, dD, dv, dx, dxn, dr, 25)
        out["jacr_x"], out["jacr_r"], out["jacr_s"] = ctx.download(dxn, n), ctx.download(dr, n), ctx.scalars(25)[0]
    finally:
        for d in (dx, dv, dD, dy, dr, dt, dxn):
            ctx.free(d)
    return out


# ---- b: Anderson past 2^31, more than 256 distinct values --------------------------------------------------
ANDERSON = dict(lx=700, ly=700, lz=630, ranpot=5.0, t=1.0, seed=1)


@pytest.fixture(scope="class", params=["open", "periodic"])
def anderson(ctx, request):
    periodic = request.param == "periodic"
    a = ANDERSON
    need(ctx, 35, "Anderson 700 x 700 x 630 (CRS 28 GB, window format 4 GB)")
    with options(ctx, spmv_variant=0):
        A = ctx.generate_anderson(a["lx"], a["ly"], a["lz"], a["ranpot"], a["t"], a["seed"], periodic)
    slabs = port.anderson_slabs(a["lx"], a["ly"], a["lz"], PLANES, a["ranpot"], a["t"], a["seed"], periodic)
    try:
        yield SimpleNamespace(A=A, n=slabs.n, slabs=slabs, periodic=periodic)
    finally:
        A.free()


class TestAnderson:
    def test_generator_limit_is_the_column_id(self, ctx):
        """2^31 sites would overflow the 32-bit column ids: refused before anything is allocated"""
        with pytest.raises(capi.BisError, match="exceed 32-bit column ids"):
            ctx.generate_anderson(1024, 1024, 2048)

    def test_spmv(self, ctx, anderson):
        A, n = anderson.A, anderson.n
        inf = A.info()
        assert inf["nnz"] == (2_160_900_000 if anderson.periodic else 2_158_156_000) and inf["nnz"] >= INT31
        assert inf["rp_bytes"] == 8
        x = np.random.default_rng(61).uniform(-1.0, 1.0, n)
        y_ref = port.spmv_slabwise(anderson.slabs, x)
        dx = ctx.upload(x)
        try:
            if not anderson.periodic:
                for variant in (3, 2):
                    with options(ctx, spmv_variant=variant):
                        assert_bits(spmv(ctx, A, dx, n), y_ref, f"open, variant {variant}")
                        if variant == 3:
                            assert ctx.get_option("spmv_value_bytes") == 8    # more than 256 values: no dictionary
            else:
                with options(ctx, spmv_variant=0):
                    y = spmv(ctx, A, dx, n)
                # auto takes the windowed variant whenever it can (x is aligned): ask it whether it can
                with options(ctx, spmv_variant=3):
                    try:
                        y3 = spmv(ctx, A, dx, n)
                        taken = 3
                    except capi.BisError as e:
                        assert "spmv_variant=3 forced" in str(e), e
                        y3, taken = y_ref, 2
                assert_bits(y, y_ref, f"periodic, auto (variant {taken})")
                assert_bits(y3, y_ref, "periodic, variant 3")
        finally:
            ctx.free(dx)


# ---- c: SpMM with n*k > 2^31 -------------------------------------------------------------------------------
SPMM_DIMS = (512, 512, 520)


@pytest.fixture(scope="class")
def hpcg_spmm(ctx):
    nx, ny, nz = SPMM_DIMS
    need(ctx, 125, "HPCG 512 x 512 x 520 (56 GB) and the SpMM blocks (65 GB)")
    with options(ctx, spmv_variant=0, spmv_vdict=1):
        A = ctx.generate_hpcg(nx, ny, nz)
    try:
        yield SimpleNamespace(A=A, n=nx * ny * nz, slabs=port.hpcg_slabs(nx, ny, nz, PLANES))
    finally:
        A.free()


class TestSpmm:
    def test_spmm_columns(self, ctx, hpcg_spmm):
        """column j of Y = A X is the oracle's SpMV of column j, bit for bit, for k = 1, 3, 16 (n*k > 2^31)"""
        import torch
        A, n = hpcg_spmm.A, hpcg_spmm.n
        inf = A.info()
        assert inf["nnz"] == 3_666_217_048 and inf["rp_bytes"] == 8
        assert n * 16 > INT31
        ks = (1, 3, 16)
        # the blocks live only in `buf` (no other name holds them), so they are released even when a check fails
        buf = {("X", 16): torch.empty((n, 16), dtype=torch.float64, device="cuda")}
        try:
            for j in range(16):
                buf["X", 16][:, j].copy_(torch.from_numpy(np.random.default_rng(700 + j).uniform(-1.0, 1.0, n)))
            buf["X", 3] = buf["X", 16][:, :3].contiguous()
            buf["X", 1] = buf["X", 16][:, :1].contiguous()
            for vdict in (1, 0):
                with options(ctx, spmv_vdict=vdict):
                    for k in ks:
                        buf["Y", vdict, k] = torch.full((n, k), float("nan"), dtype=torch.float64, device="cuda")
                        torch.cuda.synchronize()        # torch fills on its stream, the library runs on its own
                        ctx.spmm(A, buf["X", k].data_ptr(), buf["Y", vdict, k].data_ptr(), k)
                        ctx.sync()
            track(ctx)
            for j in range(16):
                y_ref = port.spmv_slabwise(hpcg_spmm.slabs, column(buf["X", 16], j))
                for vdict in (1, 0):
                    for k in ks:
                        if j < k:
                            assert_bits(column(buf["Y", vdict, k], j), y_ref, f"k = {k}, vdict = {vdict}, column {j}")
        finally:
            buf.clear()
            torch.cuda.empty_cache()


# ---- d: block streaming kernels with n*k > 2^31 ------------------------------------------------------------
K = 16
FROZEN = 5                                   # the column whose state says it has stopped
S_OUT_A, S_OUT_B, S_RZ, S_PAP, S_RZN = 20, 40, 60, 80, 100


@pytest.fixture(scope="class")
def blocks(ctx):
    """three input blocks of small integers, a diagonal of powers of two, three output blocks (105 GB)"""
    import torch
    nx, ny, nz = SPMM_DIMS
    n = nx * ny * nz
    need(ctx, 110, "six n x 16 blocks")
    g = torch.Generator(device="cuda")
    g.manual_seed(81)
    ins = [torch.randint(-8, 9, (n, K), generator=g, dtype=torch.float64, device="cuda") for _ in range(3)]
    D = torch.pow(2.0, torch.randint(0, 3, (n,), generator=g, dtype=torch.float64, device="cuda"))
    outs = [torch.empty((n, K), dtype=torch.float64, device="cuda") for _ in range(3)]
    state = torch.zeros(3 * K, dtype=torch.float64, device="cuda")
    state[K:2 * K] = 1.0
    state[K + FROZEN] = 0.0
    torch.cuda.synchronize()
    ns = SimpleNamespace(n=n, ins=ins, D=D, outs=outs, state=state)
    del ins, outs, D, state
    try:
        yield ns
    finally:
        ns.ins = ns.outs = ns.D = ns.state = None
        torch.cuda.empty_cache()


def column(t, j):
    """column j of an n x k device block, on the host"""
    return t[:, j].contiguous().cpu().numpy()


def set_slots(ctx, first, values):
    for j, v in enumerate(values):
        ctx.call("bis_scalar_set", first + j, float(v))


class TestBlockKernels:
    """Blocks are named by index (blocks.ins[i], blocks.outs[i]) and never bound to a local name, so a failing
    check does not keep 17 GB alive in its traceback."""

    def _prepare(self, ctx, blocks):
        import torch
        for o in blocks.outs:
            o.fill_(float("nan"))
        torch.cuda.synchronize()
        for s in (S_OUT_A, S_OUT_B):
            set_slots(ctx, s, [float("nan")] * K)
        # alpha_j = rz / pAp = 2^-(j % 3), beta_j = rz_new / rz = 2^-(j % 2): every product is exact
        set_slots(ctx, S_RZ, [1.0] * K)
        set_slots(ctx, S_PAP, [2.0 ** (j % 3) for j in range(K)])
        set_slots(ctx, S_RZN, [0.5 ** (j % 2) for j in range(K)])

    def _run(self, ctx, name, *args):
        import torch
        torch.cuda.synchronize()
        ctx.call(name, *args)
        ctx.sync()
        track(ctx)

    @staticmethod
    def _ptr(blocks, which, i):
        return getattr(blocks, which)[i].data_ptr()

    def test_dot_to_slots(self, ctx, blocks):
        self._prepare(ctx, blocks)
        p = lambda i: self._ptr(blocks, "ins", i)
        self._run(ctx, "bis_block_dot_to_slots", blocks.n, K, p(0), p(1), S_OUT_A, blocks.state.data_ptr())
        got = ctx.scalars(S_OUT_A, K)
        for j in range(K):
            if j == FROZEN:
                assert np.isnan(got[j]), "the frozen column's slot was written"
            else:
                a, b = column(blocks.ins[0], j).astype(np.int64), column(blocks.ins[1], j).astype(np.int64)
                assert_exact(got[j], int(a @ b), f"dot {j}")

    @pytest.mark.parametrize("precond", ["none", "j"])
    def test_residual(self, ctx, blocks, precond):
        """in: AX = ins[0], B = ins[1]; out: R, Z, P = outs (no state: every column is written)"""
        self._prepare(ctx, blocks)
        jac = precond == "j"
        i, o = (lambda k: self._ptr(blocks, "ins", k)), (lambda k: self._ptr(blocks, "outs", k))
        self._run(ctx, "bis_block_residual", capi.PRECOND[precond], blocks.n, K, i(0), i(1),
                  blocks.D.data_ptr() if jac else None, o(0), o(1), o(2), S_OUT_A, S_OUT_B)
        rz, rr = ctx.scalars(S_OUT_A, K), ctx.scalars(S_OUT_B, K)
        d = blocks.D.cpu().numpy() if jac else np.ones(blocks.n)
        q = (4 // d).astype(np.int64)           # 4 / d: r*z = r^2 * q / 4 exactly
        for j in range(K):
            r = column(blocks.ins[1], j) - column(blocks.ins[0], j)
            z = r / (1.0 * d)
            assert_bits(column(blocks.outs[0], j), r, f"R {j}")
            assert_bits(column(blocks.outs[1], j), z, f"Z {j}")
            assert_bits(column(blocks.outs[2], j), z, f"P {j}")
            ri = r.astype(np.int64)
            assert_exact(rr[j], int(ri @ ri), f"rr {j}")
            assert_exact(rz[j], int((ri * ri) @ q) / 4, f"rz {j}")

    def test_cg_update(self, ctx, blocks):
        """in: R_old = ins[0], AP = ins[1]; out: R_new = outs[0], Z_new = outs[1]; Jacobi"""
        self._prepare(ctx, blocks)
        i, o = (lambda k: self._ptr(blocks, "ins", k)), (lambda k: self._ptr(blocks, "outs", k))
        self._run(ctx, "bis_block_cg_update", capi.PRECOND["j"], blocks.n, K, o(0), i(0), i(1), o(1),
                  blocks.D.data_ptr(), S_RZ, S_PAP, S_OUT_A, S_OUT_B, blocks.state.data_ptr())
        rr, rz = ctx.scalars(S_OUT_A, K), ctx.scalars(S_OUT_B, K)
        d = blocks.D.cpu().numpy()
        q = (4 // d).astype(np.int64)
        for j in range(K):
            if j == FROZEN:
                assert np.all(np.isnan(column(blocks.outs[0], j))), "the frozen column's R_new was written"
                assert np.all(np.isnan(column(blocks.outs[1], j))), "the frozen column's Z_new was written"
                assert np.isnan(rr[j]) and np.isnan(rz[j]), "the frozen column's slots were written"
                continue
            alpha = 1.0 / 2.0 ** (j % 3)
            r = column(blocks.ins[0], j) - alpha * column(blocks.ins[1], j)
            assert_bits(column(blocks.outs[0], j), r, f"R_new {j}")
            assert_bits(column(blocks.outs[1], j), r / d, f"Z_new {j}")
            r4 = (r * 4).astype(np.int64)         # r is a multiple of 1/4
            assert_exact(rr[j], int(r4 @ r4) / 16, f"rr {j}")
            assert_exact(rz[j], int((r4 * r4) @ q) / 64, f"rz_new {j}")

    def test_cg_direction_x(self, ctx, blocks):
        """in: Z_new = ins[0], P_old = ins[1], X_old = ins[2]; out: P_new = outs[0], X_new = outs[1]"""
        self._prepare(ctx, blocks)
        i, o = (lambda k: self._ptr(blocks, "ins", k)), (lambda k: self._ptr(blocks, "outs", k))
        self._run(ctx, "bis_block_cg_direction_x", blocks.n, K, o(0), i(0), i(1), o(1), i(2), S_RZN, S_RZ, S_PAP,
                  blocks.state.data_ptr())
        for j in range(K):
            p, x = column(blocks.ins[1], j), column(blocks.ins[2], j)
            if j == FROZEN:
                assert_bits(column(blocks.outs[1], j), x, "the frozen column's X_new = X_old")
                assert np.all(np.isnan(column(blocks.outs[0], j))), "the frozen column's P_new was written"
                continue
            alpha, beta = 1.0 / 2.0 ** (j % 3), 0.5 ** (j % 2)
            assert_bits(column(blocks.outs[1], j), x + alpha * p, f"X_new {j}")
            assert_bits(column(blocks.outs[0], j), column(blocks.ins[0], j) + beta * p, f"P_new {j}")


# ---- f: the 2^31 guard of the triangular split --------------------------------------------------------------
@pytest.fixture(scope="class")
def hpcg640(ctx):
    dims = (512, 512, 640)
    need(ctx, 62, "HPCG 512 x 512 x 640 (CRS 56 GB)")
    with options(ctx, spmv_variant=2):          # no window format: it is not what this case checks
        A = ctx.generate_hpcg(*dims)
    try:
        yield SimpleNamespace(A=A, dims=dims, n=dims[0] * dims[1] * dims[2])
    finally:
        A.free()


class TestFactorGuard:
    def test_split_refuses_a_factor_past_int32(self, ctx, hpcg640):
        A, n, (nx, ny, nz) = hpcg640.A, hpcg640.n, hpcg640.dims
        assert A.info()["nnz"] == matgen.hpcg_nnz(nx, ny, nz)
        assert (matgen.hpcg_nnz(nx, ny, nz) - n) // 2 == 2_172_790_524 > INT31 - 1
        free0 = ctx.info()["free"]
        with options(ctx, factor_keep_crs=0):
            with pytest.raises(capi.BisError, match=r"more than 2\^31-1 nonzeros"):
                ctx.split_triangular(A)
        free1 = ctx.info()["free"]
        assert abs(free1 - free0) <= (8 << 20), f"free device memory moved by {(free1 - free0) / 2**20:.1f} MB"
        # A is intact: its first and last 2 M rows against the oracle
        x = np.random.default_rng(91).uniform(-1.0, 1.0, n)
        dx = ctx.upload(x)
        try:
            with options(ctx, spmv_variant=2):
                y = spmv(ctx, A, dx, n)
        finally:
            ctx.free(dx)
        rows = 8 * nx * ny
        y_ref = np.full(n, np.nan)
        for rb in (0, n - rows):
            port.spmv_slab_into(*port.rebase(*matgen.hpcg(nx, ny, nz, rb, rb + rows), rb), x, y_ref, rb)
            assert_bits(y[rb:rb + rows], y_ref[rb:rb + rows], f"rows [{rb}, {rb + rows})")
