"""ctypes binding of the C-ABI (include/bis_b200.h -> lib/libbis_b200.so).

This is plumbing for tests and bench.py: every call goes straight through the
extern "C" boundary.  There is no CPU fallback: loading fails loudly when the
library is missing, and every call raises BisError on a non-zero status.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BIS_LIB_PATH") or os.path.join(HERE, "lib", "libbis_b200.so")   # BIS_LIB_PATH: experiment builds (tools/)
HEADER_PATH = os.path.join(os.path.dirname(HERE), "include", "bis_b200.h")

NUM_SCALARS = 128
PRECOND = {"none": 0, "j": 1, "gs": 2, "bgs": 3, "sgs": 4, "2st": 5, "s2st": 6, "ilu0": 7}

c_ctx = C.c_void_p
c_mat = C.c_void_p
c_dev = C.c_void_p      # device address of a double vector
i64 = C.c_int64
dbl = C.c_double
cint = C.c_int


class BisError(RuntimeError):
    pass


_SIGS = {
    "bis_version": ([], cint),
    "bis_device_count": ([C.POINTER(cint)], cint),
    "bis_context_create": ([cint, C.POINTER(c_ctx)], cint),
    "bis_context_create_distributed": ([cint, cint, cint, C.c_void_p, C.c_size_t, C.POINTER(c_ctx)], cint),
    "bis_nccl_unique_id": ([C.c_void_p, C.c_size_t], cint),
    "bis_context_destroy": ([c_ctx], cint),
    "bis_context_synchronize": ([c_ctx], cint),
    "bis_context_rank": ([c_ctx, C.POINTER(cint), C.POINTER(cint)], cint),
    "bis_context_info": ([c_ctx, C.POINTER(i64)], cint),
    "bis_timer_start": ([c_ctx], cint),
    "bis_timer_stop": ([c_ctx, C.POINTER(dbl)], cint),
    "bis_flush_l2": ([c_ctx], cint),
    "bis_profile_enable": ([c_ctx, cint], cint),
    "bis_profile_read": ([c_ctx, C.c_char_p, C.POINTER(dbl), C.POINTER(i64)], cint),
    "bis_context_set_option": ([c_ctx, C.c_char_p, cint], cint),
    "bis_context_get_option": ([c_ctx, C.c_char_p, C.POINTER(cint)], cint),
    "bis_graph_begin": ([c_ctx], cint),
    "bis_graph_end": ([c_ctx, C.POINTER(C.c_void_p)], cint),
    "bis_graph_abort": ([c_ctx], cint),
    "bis_graph_launch": ([c_ctx, C.c_void_p], cint),
    "bis_graph_free": ([c_ctx, C.c_void_p], cint),
    "bis_dist_wait_read": ([c_ctx, C.POINTER(dbl), cint], cint),
    "bis_dist_stream_barrier": ([c_ctx], cint),
    "bis_partition_row_block": ([i64, i64, cint, cint, C.POINTER(i64), C.POINTER(i64)], cint),
    "bis_vector_alloc": ([c_ctx, i64, C.POINTER(c_dev)], cint),
    "bis_vector_free": ([c_ctx, c_dev], cint),
    "bis_vector_upload": ([c_ctx, c_dev, C.c_void_p, i64], cint),
    "bis_vector_download": ([c_ctx, C.c_void_p, c_dev, i64], cint),
    "bis_matrix_upload_crs": ([c_ctx, i64, i64, i64, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(c_mat)], cint),
    "bis_matrix_upload_crs64": ([c_ctx, i64, i64, i64, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(c_mat)], cint),
    "bis_matrix_upload_coo": ([c_ctx, i64, i64, i64, C.c_void_p, C.c_void_p, C.c_void_p, cint, C.POINTER(c_mat)], cint),
    "bis_matrix_upload_crs_distributed": ([c_ctx, i64, i64, i64, i64, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(c_mat)], cint),
    "bis_matrix_upload_triangular": ([c_ctx, i64, i64, C.c_void_p, C.c_void_p, C.c_void_p, cint, C.POINTER(c_mat)], cint),
    "bis_matrix_generate_hpcg": ([c_ctx, cint, cint, cint, C.POINTER(c_mat)], cint),
    "bis_matrix_generate_anderson": ([c_ctx, cint, cint, cint, dbl, dbl, C.c_uint64, cint, C.POINTER(c_mat)], cint),
    "bis_matrix_free": ([c_ctx, c_mat], cint),
    "bis_matrix_info": ([c_mat, C.POINTER(i64)], cint),
    "bis_matrix_download_crs": ([c_ctx, c_mat, C.c_void_p, C.c_void_p, C.c_void_p], cint),
    "bis_matrix_extract_diagonal": ([c_ctx, c_mat, c_dev, c_dev], cint),
    "bis_matrix_split_triangular": ([c_ctx, c_mat, C.POINTER(c_mat), C.POINTER(c_mat)], cint),
    "bis_matrix_scale_symmetric": ([c_ctx, c_mat, c_dev], cint),
    "bis_matrix_colouring_permutation": ([c_ctx, c_mat, C.c_void_p, C.c_void_p, C.POINTER(cint)], cint),
    "bis_matrix_bfs_permutation": ([c_ctx, c_mat, cint, C.c_void_p, C.c_void_p, C.POINTER(cint)], cint),
    "bis_matrix_permute_symmetric": ([c_ctx, c_mat, C.c_void_p, C.c_void_p, C.POINTER(c_mat)], cint),
    "bis_vector_permute": ([c_ctx, c_dev, c_dev, C.c_void_p, i64], cint),
    "bis_index_alloc": ([c_ctx, i64, C.POINTER(C.c_void_p)], cint),
    "bis_index_free": ([c_ctx, C.c_void_p], cint),
    "bis_index_download": ([c_ctx, C.c_void_p, C.c_void_p, i64], cint),
    "bis_matrix_ilu0": ([c_ctx, c_mat, C.c_double, C.c_double, C.POINTER(c_mat), C.POINTER(c_mat), c_dev, c_dev], cint),
    "bis_spmv": ([c_ctx, c_mat, c_dev, c_dev], cint),
    "bis_sptrsv": ([c_ctx, c_mat, c_dev, c_dev, c_dev], cint),
    "bis_bsptrsv": ([c_ctx, c_mat, c_dev, c_dev, c_dev], cint),
    "bis_subtract_vectors": ([c_ctx, c_dev, c_dev, c_dev, i64, dbl], cint),
    "bis_sum_vectors": ([c_ctx, c_dev, c_dev, c_dev, i64, dbl], cint),
    "bis_elemwise_mult_vectors": ([c_ctx, c_dev, c_dev, c_dev, i64, dbl], cint),
    "bis_elemwise_div_vectors": ([c_ctx, c_dev, c_dev, c_dev, i64, dbl], cint),
    "bis_compute_residual": ([c_ctx, c_mat, c_dev, c_dev, c_dev, c_dev], cint),
    "bis_euclidean_vec_norm": ([c_ctx, c_dev, i64, C.POINTER(dbl)], cint),
    "bis_dot": ([c_ctx, c_dev, c_dev, i64, C.POINTER(dbl)], cint),
    "bis_scale": ([c_ctx, c_dev, c_dev, dbl, i64], cint),
    "bis_init_vector": ([c_ctx, c_dev, dbl, i64], cint),
    "bis_copy_vector": ([c_ctx, c_dev, c_dev, i64], cint),
    "bis_normalize_x": ([c_ctx, c_dev, c_dev, c_dev, c_dev, i64], cint),
    "bis_apply_preconditioner": ([c_ctx, cint, i64, c_mat, c_mat] + [c_dev] * 8, cint),
    "bis_scalar_set": ([c_ctx, cint, dbl], cint),
    "bis_scalar_get": ([c_ctx, cint, cint, C.POINTER(dbl)], cint),
    "bis_scalar_read_begin": ([c_ctx, cint, cint], cint),
    "bis_scalar_read_end": ([c_ctx, cint, cint, C.POINTER(dbl)], cint),
    "bis_scalar_copy": ([c_ctx, cint, cint], cint),
    "bis_dot_to_slot": ([c_ctx, c_dev, c_dev, i64, cint], cint),
    "bis_sumsq_to_slot": ([c_ctx, c_dev, i64, cint], cint),
    "bis_spmv_dot": ([c_ctx, c_mat, c_dev, c_dev, c_dev, cint, cint], cint),
    "bis_spmv_residual": ([c_ctx, c_mat, c_dev, c_dev, c_dev, c_dev, cint], cint),
    "bis_spmv_jacobi": ([c_ctx, c_mat, c_dev, c_dev, c_dev, c_dev], cint),
    "bis_spmv_jacobi_residual": ([c_ctx, c_mat, c_dev, c_dev, c_dev, c_dev, c_dev, cint], cint),
    "bis_spmv_sub": ([c_ctx, c_mat, c_dev, c_dev, c_dev], cint),
    "bis_spmv_two_stage": ([c_ctx, c_mat, c_dev, c_dev, c_dev, c_dev], cint),
    "bis_cg_update": ([c_ctx, cint, i64] + [c_dev] * 8 + [cint] * 4, cint),
    "bis_cg_direction": ([c_ctx, i64, c_dev, c_dev, c_dev, cint, cint], cint),
    "bis_cg_direction_x": ([c_ctx, i64, c_dev, c_dev, c_dev, c_dev, c_dev, cint, cint, cint], cint),
    "bis_bicgstab_s": ([c_ctx, cint, i64] + [c_dev] * 5 + [cint] * 2, cint),
    "bis_bicgstab_xr": ([c_ctx, i64] + [c_dev] * 9 + [cint] * 6, cint),
    "bis_bicgstab_p": ([c_ctx, cint, i64] + [c_dev] * 7 + [cint] * 5, cint),
    "bis_mgs_step": ([c_ctx, i64, c_dev, c_dev, c_dev, cint, cint], cint),
    "bis_scale_inv_norm": ([c_ctx, i64, c_dev, c_dev, cint], cint),
    "bis_gmres_update_x": ([c_ctx, i64, cint, c_dev, C.c_void_p, c_dev, c_dev, c_dev], cint),
    "bis_spmm": ([c_ctx, c_mat, cint, c_dev, c_dev], cint),
    "bis_block_dot_to_slots": ([c_ctx, i64, cint, c_dev, c_dev, cint, c_dev], cint),
    "bis_block_residual": ([c_ctx, cint, i64, cint] + [c_dev] * 6 + [cint] * 2, cint),
    "bis_block_cg_update": ([c_ctx, cint, i64, cint] + [c_dev] * 5 + [cint] * 4 + [c_dev], cint),
    "bis_block_cg_direction_x": ([c_ctx, i64, cint] + [c_dev] * 5 + [cint] * 3 + [c_dev], cint),
    "bis_block_cg_status": ([c_ctx, cint, cint, cint, c_dev], cint),
}

_lib = None


def declared_symbols() -> list[str]:
    """Every entry point include/bis_b200.h declares (parsed from the header)."""
    import re
    with open(HEADER_PATH) as f:
        txt = f.read()
    return sorted(set(re.findall(r"\b(bis_[a-z0-9_]+)\s*\(", txt)))


def _preload_nccl() -> None:
    """libbis_b200.so needs libnccl.so.2.  PyTorch bundles a newer NCCL under the same SONAME
    than the system one; whichever is loaded first serves the whole process, so load the
    bundled one first (when present) to keep a later `import torch` working."""
    import importlib.util
    try:
        spec = importlib.util.find_spec("nvidia")
    except (ImportError, ValueError):
        spec = None
    for base in (list(spec.submodule_search_locations) if spec and spec.submodule_search_locations else []):
        cand = os.path.join(base, "nccl", "lib", "libnccl.so.2")
        if os.path.exists(cand):
            C.CDLL(cand, mode=C.RTLD_GLOBAL)
            return


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BisError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
                       f"g.build()'` (there is no CPU fallback)")
    _preload_nccl()
    lib = C.CDLL(LIB_PATH)
    lib.bis_last_error.restype = C.c_char_p
    lib.bis_last_error.argtypes = []
    for name, (args, res) in _SIGS.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = res
    _lib = lib
    return lib


def partition_row_block(n_global: int, plane: int, rank: int, nranks: int):
    """Row block of `rank` (bis_partition_row_block: pure function of the C-ABI, no device needed)."""
    lib = load()
    b, e = i64(0), i64(0)
    if lib.bis_partition_row_block(int(n_global), int(plane), int(rank), int(nranks), C.byref(b), C.byref(e)) != 0:
        raise BisError(lib.bis_last_error().decode(errors="replace"))
    return int(b.value), int(e.value)


def check(rc: int) -> None:
    if rc != 0:
        raise BisError(f"[{rc}] {load().bis_last_error().decode(errors='replace')}")


def _np_ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Matrix:
    def __init__(self, ctx: "Context", handle):
        self.ctx, self.h = ctx, handle

    def info(self):
        arr = (i64 * 8)()
        check(load().bis_matrix_info(self.h, arr))
        keys = ["n_rows", "n_rows_global", "nnz", "nnz_global", "rp_bytes", "n_levels", "n_ghost", "row_begin"]
        return dict(zip(keys, [int(v) for v in arr]))

    def download(self):
        inf = self.info()
        rp = np.zeros(inf["n_rows"] + 1, np.int64)
        col = np.zeros(max(inf["nnz"], 1), np.int32)
        val = np.zeros(max(inf["nnz"], 1), np.float64)
        check(load().bis_matrix_download_crs(self.ctx.h, self.h, _np_ptr(rp), _np_ptr(col), _np_ptr(val)))
        return rp, col[:inf["nnz"]], val[:inf["nnz"]]

    def spmv_bytes(self):
        """Algorithmic bytes of one y = A x (SURVEY.md 8(d))."""
        inf = self.info()
        return 12 * inf["nnz"] + inf["rp_bytes"] * (inf["n_rows"] + 1) + 16 * inf["n_rows"]

    def free(self):
        if self.h:
            load().bis_matrix_free(self.ctx.h, self.h)
            self.h = None


class Context:
    """Thin OO veneer: device vectors are plain ints (device addresses)."""

    def __init__(self, device: int = 0, rank: int = 0, nranks: int = 1, nccl_id: bytes | None = None):
        lib = load()
        h = c_ctx()
        if nranks > 1:
            buf = C.create_string_buffer(nccl_id, len(nccl_id))
            check(lib.bis_context_create_distributed(device, rank, nranks, buf, len(nccl_id), C.byref(h)))
        else:
            check(lib.bis_context_create(device, C.byref(h)))
        self.h = h
        self.lib = lib
        self.rank, self.nranks = rank, nranks

    @staticmethod
    def nccl_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        check(load().bis_nccl_unique_id(buf, 128))
        return buf.raw

    def close(self):
        if self.h:
            self.lib.bis_context_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def call(self, name, *args):
        check(getattr(self.lib, name)(self.h, *args))

    def sync(self):
        self.call("bis_context_synchronize")

    def info(self):
        arr = (i64 * 8)()
        self.call("bis_context_info", arr)
        return {"sm_count": int(arr[0]), "free": int(arr[1]), "total": int(arr[2]),
                "launches": int(arr[3]), "l2_bytes": int(arr[4]),
                "peer_memory": bool(arr[5]), "chain_solves": int(arr[6]), "wave_solves": int(arr[7])}

    def set_option(self, key: str, value: int):
        self.call("bis_context_set_option", key.encode(), int(value))

    def get_option(self, key: str) -> int:
        v = cint(0)
        self.call("bis_context_get_option", key.encode(), C.byref(v))
        return int(v.value)

    # vectors -----------------------------------------------------------------
    def alloc(self, n: int) -> int:
        p = c_dev()
        self.call("bis_vector_alloc", n, C.byref(p))
        return p.value

    def free(self, v: int):
        self.call("bis_vector_free", v)

    def upload(self, host: np.ndarray, dev: int | None = None) -> int:
        host = np.ascontiguousarray(host, dtype=np.float64)
        if dev is None:
            dev = self.alloc(host.size)
        self.call("bis_vector_upload", dev, _np_ptr(host), host.size)
        return dev

    def download(self, dev: int, n: int) -> np.ndarray:
        out = np.empty(n, np.float64)
        self.call("bis_vector_download", _np_ptr(out), dev, n)
        return out

    # matrices ----------------------------------------------------------------
    def upload_crs(self, rp, col, val, n_cols=None) -> Matrix:
        col = np.ascontiguousarray(col, dtype=np.int32)
        val = np.ascontiguousarray(val, dtype=np.float64)
        n = len(rp) - 1
        m = c_mat()
        if np.asarray(rp).dtype == np.int64:
            rp = np.ascontiguousarray(rp, dtype=np.int64)
            self.call("bis_matrix_upload_crs64", n, n if n_cols is None else n_cols, int(rp[-1]),
                      _np_ptr(rp), _np_ptr(col), _np_ptr(val), C.byref(m))
        else:
            rp = np.ascontiguousarray(rp, dtype=np.int32)
            self.call("bis_matrix_upload_crs", n, n if n_cols is None else n_cols, int(rp[-1]),
                      _np_ptr(rp), _np_ptr(col), _np_ptr(val), C.byref(m))
        return Matrix(self, m)

    def bfs_permutation(self, A: Matrix, mode: int):
        """(perm, inv_perm, n_levels): mode 2 = BFS levels, 3 = reverse Cuthill-McKee, 4 = Cuthill-McKee (host arrays)."""
        n = A.info()["n_rows"]
        dp, di = C.c_void_p(), C.c_void_p()
        self.call("bis_index_alloc", n, C.byref(dp))
        self.call("bis_index_alloc", n, C.byref(di))
        nl = cint(0)
        self.call("bis_matrix_bfs_permutation", A.h, mode, dp, di, C.byref(nl))
        perm, inv = np.zeros(n, np.int32), np.zeros(n, np.int32)
        self.call("bis_index_download", _np_ptr(perm), dp, n)
        self.call("bis_index_download", _np_ptr(inv), di, n)
        self.call("bis_index_free", dp)
        self.call("bis_index_free", di)
        return perm, inv, int(nl.value)

    def colouring_permutation(self, A: Matrix):
        """(perm, inv_perm, n_colours) of the multicolouring permutation of A (host arrays)."""
        n = A.info()["n_rows"]
        dp, di = C.c_void_p(), C.c_void_p()
        self.call("bis_index_alloc", n, C.byref(dp))
        self.call("bis_index_alloc", n, C.byref(di))
        nc = cint(0)
        self.call("bis_matrix_colouring_permutation", A.h, dp, di, C.byref(nc))
        perm, inv = np.zeros(n, np.int32), np.zeros(n, np.int32)
        self.call("bis_index_download", _np_ptr(perm), dp, n)
        self.call("bis_index_download", _np_ptr(inv), di, n)
        self.call("bis_index_free", dp)
        self.call("bis_index_free", di)
        return perm, inv, int(nc.value)

    def upload_coo(self, n_rows, n_cols, I, J, V, sorted_by_row=False) -> Matrix:
        I = np.ascontiguousarray(I, np.int32)
        J = np.ascontiguousarray(J, np.int32)
        V = np.ascontiguousarray(V, np.float64)
        h = c_mat()
        self.call("bis_matrix_upload_coo", int(n_rows), int(n_cols), int(V.size), _np_ptr(I), _np_ptr(J), _np_ptr(V),
                  int(sorted_by_row), C.byref(h))
        return Matrix(self, h)

    def upload_crs_distributed(self, row_begin, n_global, rp, col, val) -> Matrix:
        rp = np.ascontiguousarray(rp, dtype=np.int64)
        col = np.ascontiguousarray(col, dtype=np.int32)
        val = np.ascontiguousarray(val, dtype=np.float64)
        m = c_mat()
        self.call("bis_matrix_upload_crs_distributed", int(row_begin), len(rp) - 1, int(n_global),
                  int(rp[-1]), _np_ptr(rp), _np_ptr(col), _np_ptr(val), C.byref(m))
        return Matrix(self, m)

    def upload_triangular(self, rp, col, val, upper: bool) -> Matrix:
        rp = np.ascontiguousarray(rp, dtype=np.int32)
        col = np.ascontiguousarray(col, dtype=np.int32)
        val = np.ascontiguousarray(val, dtype=np.float64)
        m = c_mat()
        self.call("bis_matrix_upload_triangular", len(rp) - 1, int(rp[-1]), _np_ptr(rp), _np_ptr(col),
                  _np_ptr(val), int(upper), C.byref(m))
        return Matrix(self, m)

    def generate_hpcg(self, nx, ny=None, nz=None) -> Matrix:
        m = c_mat()
        self.call("bis_matrix_generate_hpcg", nx, nx if ny is None else ny, nx if nz is None else nz, C.byref(m))
        return Matrix(self, m)

    def generate_anderson(self, lx, ly, lz, ranpot=5.0, t=1.0, seed=1, periodic=False) -> Matrix:
        m = c_mat()
        self.call("bis_matrix_generate_anderson", lx, ly, lz, float(ranpot), float(t), int(seed),
                  int(periodic), C.byref(m))
        return Matrix(self, m)

    def split_triangular(self, A: Matrix):
        l, u = c_mat(), c_mat()
        self.call("bis_matrix_split_triangular", A.h, C.byref(l), C.byref(u))
        return Matrix(self, l), Matrix(self, u)

    def spmm(self, A: Matrix, X: int, Y: int, k: int):
        """Y = A X for k right-hand sides (bis_spmm): X, Y device blocks of n x k doubles, row-major."""
        self.call("bis_spmm", A.h, int(k), X, Y)

    # scalars -----------------------------------------------------------------
    def ilu0(self, A: Matrix, n: int, pivot_tolerance: float = 1e-8, pivot_replacement: float = 1e-4):
        """Device ILU(0): returns (L_strict, U_strict, L_D, U_D) with L_D/U_D device vectors."""
        l, u = c_mat(), c_mat()
        ld, ud = self.alloc(n), self.alloc(n)
        self.call("bis_matrix_ilu0", A.h, pivot_tolerance, pivot_replacement, C.byref(l), C.byref(u), ld, ud)
        return Matrix(self, l), Matrix(self, u), ld, ud

    def scalars(self, first: int, count: int = 1) -> np.ndarray:
        arr = (dbl * count)()
        self.call("bis_scalar_get", first, count, arr)
        return np.array(arr[:], dtype=np.float64)

    def dot(self, a: int, b: int, n: int) -> float:
        r = dbl()
        self.call("bis_dot", a, b, n, C.byref(r))
        return r.value

    def norm(self, v: int, n: int) -> float:
        r = dbl()
        self.call("bis_euclidean_vec_norm", v, n, C.byref(r))
        return r.value

    # timing ------------------------------------------------------------------
    def dist_wait_read(self, reset: bool = False):
        """In-kernel wait accounting of a distributed context (bis_dist_wait_read), ns."""
        out = (dbl * 4)()
        check(load().bis_dist_wait_read(self.h, out, int(reset)))
        return [float(v) for v in out]

    def profile_enable(self, on: bool = True):
        self.call("bis_profile_enable", int(on))

    def profile_read(self, family: str):
        ms, cnt = dbl(), i64()
        self.call("bis_profile_read", family.encode(), C.byref(ms), C.byref(cnt))
        return ms.value, int(cnt.value)

    def timer_start(self):
        self.call("bis_timer_start")

    def timer_stop(self) -> float:
        ms = dbl()
        self.call("bis_timer_stop", C.byref(ms))
        return ms.value
