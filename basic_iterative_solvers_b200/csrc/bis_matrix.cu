// bis_matrix.cu -- device CRS containers (MatrixCRS, sparse_matrix.hpp:59-179),
// level sets for the strictly triangular factors, device-side synthetic
// generators (SURVEY.md 8(d)), row partitioning + halo index lists.
#include "bis_device.cuh"

#include <thrust/copy.h>
#include <thrust/device_ptr.h>
#include <thrust/execution_policy.h>
#include <thrust/iterator/zip_iterator.h>
#include <thrust/tuple.h>
#include <thrust/scan.h>
#include <thrust/sort.h>
#include <thrust/unique.h>

#include <algorithm>
#include <cstring>
#include <numeric>

namespace {

template <typename T> int dev_alloc(T **p, size_t count) {
    BIS_CUDA(bis_cuda_malloc(p, sizeof(T) * (count > 0 ? count : 1)));
    return 0;
}

void free_matrix_storage(bis_matrix *A) {
    cudaFree(A->d_rp);
    cudaFree(A->d_col);
    cudaFree(A->d_val);
    cudaFree(A->lv.d_slot_row);
    cudaFree(A->lv.d_slot_level);
    cudaFree(A->lv.d_level);
    cudaFree(A->lv.chain.d_recs);
    cudaFree(A->lv.chain.d_slice_off);
    cudaFree(A->lv.chain.d_w);
    cudaFree(A->lv.d_slot_gate);
    cudaFree(A->lv.d_level_size);
    cudaFree(A->lv.d_level_done);
    cudaFree(A->lv.d_ticket);
    cudaFree(A->lv.d_w);
    cudaFree(A->lv.d_w2);
    cudaFree(A->lv.d_bw[0]);
    cudaFree(A->lv.d_bw[1]);
    cudaFree(A->lv.wave.d_rec);
    cudaFree(A->lv.wave.d_w[0]);
    cudaFree(A->lv.wave.d_w[1]);
    cudaFree(A->lv.wave.d_ticket);
    cudaFree(A->lv.d_rp);
    cudaFree(A->lv.d_col);
    cudaFree(A->lv.d_val);
    cudaFree(A->halo.d_ghost);
    cudaFree(A->halo.d_sendbuf);
    cudaFree(A->halo.d_send_idx);
    cudaFree(A->halo.d_ghost_global);
    cudaFree(A->win.d_seg_start);
    cudaFree(A->win.d_seg_len);
    cudaFree(A->win.d_seg_off);
    cudaFree(A->win.d_nseg);
    cudaFree(A->win.d_lidx);
    cudaFree(A->win.d_order);
    cudaFree(A->win.d_vidx);
    cudaFree(A->win.d_vdict);
    cudaFree(A->win.d_class_mask);
    cudaFree(A->win.d_row_class);
}

template <typename RP>
int upload_common(bis_context *c, int64_t n_rows, int64_t n_cols, int64_t nnz, const RP *rp,
                  const int32_t *col, const double *val, bis_matrix **out) {
    BIS_REQUIRE(c && out && rp, "matrix upload: null argument");
    BIS_REQUIRE(n_rows >= 0 && n_cols >= 0 && nnz >= 0, "matrix upload: negative size");
    BIS_REQUIRE(nnz == 0 || (col && val), "matrix upload: null col/val");
    BIS_REQUIRE((int64_t)rp[n_rows] == nnz, "matrix upload: row_ptr[n_rows]=%lld != nnz=%lld",
                (long long)rp[n_rows], (long long)nnz);
    BIS_REQUIRE(n_rows < INT32_MAX && n_cols < INT32_MAX, "matrix upload: more than 2^31-1 rows");
    BIS_CUDA(cudaSetDevice(c->device));
    bis_vector_cache_trim(c);
    bis_matrix *A = new bis_matrix;
    A->n_rows = n_rows;
    A->n_cols = n_cols;
    A->n_rows_global = n_rows;
    A->nnz = A->nnz_global = nnz;
    A->rp_bytes = (int)sizeof(RP);
    int max_row = 0;
    for (int64_t r = 0; r < n_rows; ++r) {
        int64_t len = (int64_t)rp[r + 1] - (int64_t)rp[r];
        if (len < 0) {
            bis_set_error("matrix upload: row_ptr not monotone at row %lld", (long long)r);
            delete A;
            return 2;
        }
        if (len > max_row) max_row = (int)len;
    }
    A->max_row = max_row;
    A->mean_row = n_rows ? (double)nnz / (double)n_rows : 0.0;
    RP *d_rp = nullptr;
    if (dev_alloc(&d_rp, (size_t)n_rows + 1 + 8) || dev_alloc(&A->d_col, (size_t)nnz + 8) ||
        dev_alloc(&A->d_val, (size_t)nnz + 8)) {
        A->d_rp = d_rp;
        free_matrix_storage(A);
        delete A;
        return 1;
    }
    A->d_rp = d_rp;
    BIS_CUDA(cudaMemcpyAsync(d_rp, rp, sizeof(RP) * ((size_t)n_rows + 1), cudaMemcpyHostToDevice, c->stream));
    if (nnz) {
        BIS_CUDA(cudaMemcpyAsync(A->d_col, col, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, c->stream));
        BIS_CUDA(cudaMemcpyAsync(A->d_val, val, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, c->stream));
    }
    BIS_CUDA(cudaStreamSynchronize(c->stream));   // host arrays are never retained
    *out = A;
    return 0;
}

} // namespace

extern "C" int bis_matrix_upload_crs(bis_context *c, int64_t n_rows, int64_t n_cols, int64_t nnz,
                                     const int32_t *rp, const int32_t *col, const double *val,
                                     bis_matrix **A) {
    BIS_REQUIRE(!c || c->nranks == 1,
                "bis_matrix_upload_crs: distributed context; use bis_matrix_upload_crs_distributed");
    BIS_CHECK(upload_common<int32_t>(c, n_rows, n_cols, nnz, rp, col, val, A));
    bis_partition_set(c, n_rows, 0, 0, n_rows);
    return bis_spmv_prepare(c, *A);
}

extern "C" int bis_matrix_upload_crs64(bis_context *c, int64_t n_rows, int64_t n_cols, int64_t nnz,
                                       const int64_t *rp, const int32_t *col, const double *val,
                                       bis_matrix **A) {
    BIS_REQUIRE(!c || c->nranks == 1,
                "bis_matrix_upload_crs64: distributed context; use bis_matrix_upload_crs_distributed");
    BIS_CHECK(upload_common<int64_t>(c, n_rows, n_cols, nnz, rp, col, val, A));
    bis_partition_set(c, n_rows, 0, 0, n_rows);
    return bis_spmv_prepare(c, *A);
}

extern "C" int bis_matrix_upload_crs_distributed(bis_context *c, int64_t row_begin,
                                                 int64_t n_rows_local, int64_t n_rows_global,
                                                 int64_t nnz_local, const int64_t *rp,
                                                 const int32_t *col, const double *val,
                                                 bis_matrix **out) {
    BIS_REQUIRE(c && out, "null argument");
    bis_matrix *A = nullptr;
    BIS_CHECK(upload_common<int64_t>(c, n_rows_local, n_rows_local, nnz_local, rp, col, val, &A));
    A->n_rows_global = n_rows_global;
    A->row_begin = row_begin;
    bis_partition_set(c, n_rows_global, 0, row_begin, n_rows_local);
    if (bis_matrix_finalize_distributed(c, A, A->d_col) != 0) {
        free_matrix_storage(A);
        delete A;
        return 1;
    }
    *out = A;
    return bis_spmv_prepare(c, A);
}

// ---- COO -> CRS on the device (convert_coo_to_crs, utilities/utilities.hpp:326-367) -----------------------
// The reference's reader sorts the entries by row with a STABLE sort (sort_perm, sparse_matrix.hpp:20-30,
// :332-344) and convert_coo_to_crs counts rows: inside a row the entries keep their order of appearance in the
// file, which is the summation order of every kernel.  Same here: stable sort by row of (col, val), then
// row_ptr by binary search.  `sorted` != 0: the entries are already grouped by row (the reference's is_sorted).
namespace {
__global__ void coo_row_ptr_kernel(int64_t n_rows, int64_t nnz, const int *I, int *rp32, int64_t *rp64, int *bad) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r <= n_rows; r += (int64_t)gridDim.x * blockDim.x) {
        int64_t lo = 0, hi = nnz;     // first entry with I >= r
        while (lo < hi) {
            const int64_t m = (lo + hi) >> 1;
            if (I[m] < r) lo = m + 1;
            else hi = m;
        }
        if (rp32) rp32[r] = (int)lo;
        else rp64[r] = lo;
    }
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x) {
        if (I[k] < 0 || I[k] >= n_rows) atomicExch(bad, 1);
        if (k > 0 && I[k - 1] > I[k]) atomicExch(bad, 2);
    }
}
} // namespace

namespace {
template <typename RP> __global__ void max_row_kernel(int64_t n, const RP *rp, int *out) {
    int m = 0;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x)
        m = max(m, (int)(rp[r + 1] - rp[r]));
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}
} // namespace

// max_row / mean_row of a device CRS (what the SpMV planners look at)
int bis_matrix_stats(bis_context *c, bis_matrix *A) {
    BIS_REQUIRE_CRS(A);
    int *d_m = nullptr;
    BIS_CHECK(dev_alloc(&d_m, 1));
    BIS_CUDA(cudaMemsetAsync(d_m, 0, sizeof(int), c->stream));
    const int blocks = bis_blocks_for(A->n_rows, 256, c->sm_count * 8);
    if (A->rp_bytes == 8) max_row_kernel<int64_t><<<blocks, 256, 0, c->stream>>>(A->n_rows, static_cast<const int64_t *>(A->d_rp), d_m);
    else max_row_kernel<int32_t><<<blocks, 256, 0, c->stream>>>(A->n_rows, static_cast<const int32_t *>(A->d_rp), d_m);
    BIS_LAUNCH_CHECK(c);
    int m = 0;
    BIS_CUDA(cudaMemcpyAsync(&m, d_m, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(d_m);
    A->max_row = m;
    A->mean_row = A->n_rows ? (double)A->nnz / (double)A->n_rows : 0.0;
    return 0;
}

extern "C" int bis_matrix_upload_coo(bis_context *c, int64_t n_rows, int64_t n_cols, int64_t nnz, const int32_t *I,
                                     const int32_t *J, const double *V, int sorted, bis_matrix **out) {
    BIS_REQUIRE(c && out, "bis_matrix_upload_coo: null argument");
    BIS_REQUIRE(c->nranks == 1, "bis_matrix_upload_coo: single-GPU contexts only");
    BIS_REQUIRE(n_rows >= 0 && n_cols >= 0 && nnz >= 0 && (nnz == 0 || (I && J && V)), "bis_matrix_upload_coo: bad argument");
    BIS_REQUIRE(n_rows < INT32_MAX && n_cols < INT32_MAX, "bis_matrix_upload_coo: more than 2^31-1 rows");
    BIS_CUDA(cudaSetDevice(c->device));
    bis_vector_cache_trim(c);
    cudaStream_t st = c->stream;
    bis_matrix *A = new bis_matrix;
    A->n_rows = n_rows;
    A->n_cols = n_cols;
    A->n_rows_global = n_rows;
    A->nnz = A->nnz_global = nnz;
    A->rp_bytes = nnz >= (int64_t)INT32_MAX ? 8 : 4;
    int *d_I = nullptr, *d_bad = nullptr;
    int rc = dev_alloc(&d_I, (size_t)nnz) | dev_alloc(&d_bad, 1) | dev_alloc(&A->d_col, (size_t)nnz + 8) | dev_alloc(&A->d_val, (size_t)nnz + 8);
    if (A->rp_bytes == 8) rc |= dev_alloc(reinterpret_cast<int64_t **>(&A->d_rp), (size_t)n_rows + 1 + 8);
    else rc |= dev_alloc(reinterpret_cast<int32_t **>(&A->d_rp), (size_t)n_rows + 1 + 8);
    auto fail = [&](int code) {
        cudaFree(d_I);
        cudaFree(d_bad);
        free_matrix_storage(A);
        delete A;
        return code;
    };
    if (rc) return fail(1);
    if (nnz) {
        if (cudaMemcpyAsync(d_I, I, sizeof(int) * (size_t)nnz, cudaMemcpyHostToDevice, st) != cudaSuccess ||
            cudaMemcpyAsync(A->d_col, J, sizeof(int) * (size_t)nnz, cudaMemcpyHostToDevice, st) != cudaSuccess ||
            cudaMemcpyAsync(A->d_val, V, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, st) != cudaSuccess) {
            bis_set_error("bis_matrix_upload_coo: upload failed: %s", cudaGetErrorString(cudaGetLastError()));
            return fail(1);
        }
        if (!sorted) {
            auto vals = thrust::make_zip_iterator(thrust::make_tuple(thrust::device_pointer_cast(A->d_col), thrust::device_pointer_cast(A->d_val)));
            thrust::stable_sort_by_key(thrust::cuda::par.on(st), thrust::device_pointer_cast(d_I), thrust::device_pointer_cast(d_I) + nnz, vals);
        }
    }
    cudaMemsetAsync(d_bad, 0, sizeof(int), st);
    coo_row_ptr_kernel<<<bis_blocks_for(std::max<int64_t>(nnz, n_rows + 1), 256, c->sm_count * 8), 256, 0, st>>>(
        n_rows, nnz, d_I, A->rp_bytes == 4 ? static_cast<int *>(A->d_rp) : nullptr,
        A->rp_bytes == 8 ? static_cast<int64_t *>(A->d_rp) : nullptr, d_bad);
    c->launches++;
    int bad = 0;
    if (cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) {
        bis_set_error("bis_matrix_upload_coo: %s", cudaGetErrorString(cudaGetLastError()));
        return fail(1);
    }
    if (bad) {
        bis_set_error(bad == 1 ? "bis_matrix_upload_coo: row index outside [0, n_rows)" : "ERROR: converting to CRS.");
        return fail(2);
    }
    cudaFree(d_I);
    cudaFree(d_bad);
    if (bis_matrix_stats(c, A) != 0) {
        free_matrix_storage(A);
        delete A;
        return 1;
    }
    bis_partition_set(c, n_rows, 0, 0, n_rows);
    *out = A;
    return bis_spmv_prepare(c, A);
}

// ---- level sets ---------------------------------------------------------------
extern "C" int bis_matrix_upload_triangular(bis_context *c, int64_t n, int64_t nnz,
                                            const int32_t *rp, const int32_t *col,
                                            const double *val, int upper, bis_matrix **out) {
    BIS_REQUIRE(c && out, "null argument");
    BIS_REQUIRE(c->nranks == 1, "triangular factors are single-GPU only (they do not shard)");
    bis_matrix *T = nullptr;
    BIS_CHECK(upload_common<int32_t>(c, n, n, nnz, rp, col, val, &T));
    T->triangular = upper ? 2 : 1;
    // validation (strictly triangular), level analysis, level-ordered copy and gates: all on the device
    if (bis_build_levels_device(c, T) != 0) {
        free_matrix_storage(T);
        delete T;
        return 2;
    }
    *out = T;
    return 0;
}

// ---- synthetic generators ---------------------------------------------------------
namespace {

// number of stencil points along one axis at coordinate k (3-point, clipped)
__host__ __device__ inline int64_t cnt3(int64_t k, int64_t n) {
    return 1 + (k > 0 ? 1 : 0) + (k + 1 < n ? 1 : 0);
}
// sum of cnt3 over coordinates < k
__host__ __device__ inline int64_t pre3(int64_t k, int64_t n) {
    if (k <= 0) return 0;
    if (n == 1) return 1;
    // k rows: first has 2, interior 3, last (index n-1) 2
    return 3 * k - 1 - (k >= n ? 1 : 0);
}
__host__ __device__ inline int64_t hpcg_prefix(int64_t row, int64_t nx, int64_t ny, int64_t nz) {
    const int64_t sx = pre3(nx, nx), sy = pre3(ny, ny);
    if (row >= nx * ny * nz) return sx * sy * pre3(nz, nz);
    const int64_t x = row % nx, y = (row / nx) % ny, z = row / (nx * ny);
    return pre3(z, nz) * sx * sy + cnt3(z, nz) * (pre3(y, ny) * sx + cnt3(y, ny) * pre3(x, nx));
}

// One block per HPCG_FILL_ROWS consecutive rows: a thread forms the (<= 27) entries of its row in shared memory at
// their positions inside the block's nonzero range, then the block streams that range out with coalesced stores
// (a thread writing its own row directly scatters 27 x 12 bytes: 90 ms at HPCG-512, this: the speed of the stores).
constexpr int HPCG_FILL_ROWS = 128;
template <typename RP>
__global__ void __launch_bounds__(HPCG_FILL_ROWS) hpcg_fill_kernel(int64_t row_begin, int64_t n_local, int64_t nx, int64_t ny,
                                                                   int64_t nz, RP *rp, int *col, double *val) {
    __shared__ double s_val[HPCG_FILL_ROWS * 27];
    __shared__ int s_col[HPCG_FILL_ROWS * 27];
    __shared__ long long s_p0;
    const int64_t base = hpcg_prefix(row_begin, nx, ny, nz);
    const int64_t n_blocks = (n_local + HPCG_FILL_ROWS - 1) / HPCG_FILL_ROWS;
    for (int64_t blk = blockIdx.x; blk < n_blocks; blk += gridDim.x) {
        const int64_t i0 = blk * HPCG_FILL_ROWS;
        const int64_t i = i0 + threadIdx.x;
        const int64_t i1 = i0 + HPCG_FILL_ROWS < n_local ? i0 + HPCG_FILL_ROWS : n_local;
        int64_t p = 0;
        if (i < i1) {
            p = hpcg_prefix(row_begin + i, nx, ny, nz) - base;
            rp[i] = (RP)p;
        }
        if (threadIdx.x == 0) s_p0 = p;
        __syncthreads();
        const int64_t p0 = s_p0;
        if (i < i1) {
            const int64_t row = row_begin + i;
            const int64_t x = row % nx, y = (row / nx) % ny, z = row / (nx * ny);
            int k = (int)(p - p0);
            for (int dz = -1; dz <= 1; ++dz) {
                if (z + dz < 0 || z + dz >= nz) continue;
                for (int dy = -1; dy <= 1; ++dy) {
                    if (y + dy < 0 || y + dy >= ny) continue;
                    for (int dx = -1; dx <= 1; ++dx) {
                        if (x + dx < 0 || x + dx >= nx) continue;
                        s_col[k] = (int)(row + (dz * ny + dy) * nx + dx);
                        s_val[k] = (dx == 0 && dy == 0 && dz == 0) ? 26.0 : -1.0;
                        ++k;
                    }
                }
            }
        }
        const int64_t p1 = hpcg_prefix(row_begin + i1, nx, ny, nz) - base;
        if (i1 == n_local && threadIdx.x == 0) rp[n_local] = (RP)p1;
        __syncthreads();
        const int m = (int)(p1 - p0);
        for (int k = threadIdx.x; k < m; k += HPCG_FILL_ROWS) {
            col[p0 + k] = s_col[k];
            val[p0 + k] = s_val[k];
        }
        __syncthreads();
    }
}

__host__ __device__ inline double splitmix_unit(uint64_t seed, uint64_t idx) {
    uint64_t z = seed + (idx + 1) * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return (double)(z >> 11) * (1.0 / 9007199254740992.0);
}

struct AndersonP {
    int64_t lx, ly, lz;
    double ranpot, t;
    uint64_t seed;
    int periodic;
};

// neighbour list of one site in ascending column order; returns the count
__device__ inline int anderson_row(const AndersonP &p, int64_t row, int64_t *cols, double *vals) {
    const int64_t x = row % p.lx, y = (row / p.lx) % p.ly, z = row / (p.lx * p.ly);
    const int dxs[7] = {0, 0, -1, 0, 1, 0, 0};
    const int dys[7] = {0, -1, 0, 0, 0, 1, 0};
    const int dzs[7] = {-1, 0, 0, 0, 0, 0, 1};
    int n = 0;
    for (int k = 0; k < 7; ++k) {
        int64_t xx = x + dxs[k], yy = y + dys[k], zz = z + dzs[k];
        bool ok = true;
        if (p.periodic) {
            if (dxs[k] && p.lx <= 2) ok = ok && xx >= 0 && xx < p.lx;
            if (dys[k] && p.ly <= 2) ok = ok && yy >= 0 && yy < p.ly;
            if (dzs[k] && p.lz <= 2) ok = ok && zz >= 0 && zz < p.lz;
            xx = (xx + p.lx) % p.lx;
            yy = (yy + p.ly) % p.ly;
            zz = (zz + p.lz) % p.lz;
        } else {
            ok = xx >= 0 && xx < p.lx && yy >= 0 && yy < p.ly && zz >= 0 && zz < p.lz;
        }
        if (!ok) continue;
        cols[n] = (zz * p.ly + yy) * p.lx + xx;
        // 2u - 1 and the scaling are exact-rounded ops, identical in numpy
        vals[n] = (k == 3) ? mul_rn(p.ranpot, sub_rn(mul_rn(2.0, splitmix_unit(p.seed, (uint64_t)row)), 1.0))
                           : -p.t;
        ++n;
    }
    // periodic wrap can break the ascending order: insertion sort (<= 7 items)
    for (int i = 1; i < n; ++i) {
        int64_t cc = cols[i];
        double vv = vals[i];
        int j = i - 1;
        while (j >= 0 && cols[j] > cc) {
            cols[j + 1] = cols[j];
            vals[j + 1] = vals[j];
            --j;
        }
        cols[j + 1] = cc;
        vals[j + 1] = vv;
    }
    return n;
}

__global__ void anderson_count_kernel(AndersonP p, int64_t row_begin, int64_t n_local, int64_t *rp) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_local;
         i += (int64_t)gridDim.x * blockDim.x) {
        int64_t cols[7];
        double vals[7];
        rp[i] = anderson_row(p, row_begin + i, cols, vals);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) rp[n_local] = 0;
}

__global__ void anderson_fill_kernel(AndersonP p, int64_t row_begin, int64_t n_local,
                                     const int64_t *rp, int *col, double *val) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_local;
         i += (int64_t)gridDim.x * blockDim.x) {
        int64_t cols[7];
        double vals[7];
        int n = anderson_row(p, row_begin + i, cols, vals);
        int64_t k = rp[i];
        for (int j = 0; j < n; ++j) {
            col[k + j] = (int)cols[j];
            val[k + j] = vals[j];
        }
    }
}

void slab(int64_t n, int rank, int nranks, int64_t plane, int64_t *begin, int64_t *end) {
    // unions of the 8 virtual slabs (bis_context.cu: bis_partition_rows)
    bis_partition_rows(n, plane, rank, nranks, begin, end);
}

int finish_generated(bis_context *c, bis_matrix *A, bis_matrix **out) {
    bis_partition_set(c, A->n_rows_global, 0, A->row_begin, A->n_rows);
    if (c->nranks > 1) {
        if (bis_matrix_finalize_distributed(c, A, A->d_col) != 0) {
            free_matrix_storage(A);
            delete A;
            return 1;
        }
    }
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    *out = A;
    return bis_spmv_prepare(c, A);
}

} // namespace

extern "C" int bis_matrix_generate_hpcg(bis_context *c, int nx, int ny, int nz, bis_matrix **out) {
    BIS_REQUIRE(c && out, "null argument");
    BIS_REQUIRE(nx >= 1 && ny >= 1 && nz >= 1, "bis_matrix_generate_hpcg: bad grid %dx%dx%d", nx, ny, nz);
    const int64_t n = (int64_t)nx * ny * nz;
    BIS_REQUIRE(n < INT32_MAX, "bis_matrix_generate_hpcg: %lld rows exceed 32-bit column ids", (long long)n);
    BIS_CUDA(cudaSetDevice(c->device));
    bis_vector_cache_trim(c);
    int64_t rb = 0, re = n;
    slab(n, c->rank, c->nranks, (int64_t)nx * ny, &rb, &re);
    const int64_t n_local = re - rb;
    const int64_t nnz_local = hpcg_prefix(re, nx, ny, nz) - hpcg_prefix(rb, nx, ny, nz);
    bis_matrix *A = new bis_matrix;
    A->n_rows = A->n_cols = n_local;
    A->n_rows_global = n;
    A->row_begin = rb;
    A->nnz = nnz_local;
    A->nnz_global = hpcg_prefix(n, nx, ny, nz);
    A->max_row = (int)(std::min(nx, 3) * std::min(ny, 3) * std::min(nz, 3));
    A->grid_nx = nx; A->grid_ny = ny; A->grid_nz = nz;
    A->mean_row = n_local ? (double)nnz_local / (double)n_local : 0.0;
    const bool wide = nnz_local >= (int64_t)INT32_MAX;
    A->rp_bytes = wide ? 8 : 4;
    int rc = 0;
    if (wide) rc |= dev_alloc(reinterpret_cast<int64_t **>(&A->d_rp), (size_t)n_local + 1 + 8);
    else rc |= dev_alloc(reinterpret_cast<int32_t **>(&A->d_rp), (size_t)n_local + 1 + 8);
    rc |= dev_alloc(&A->d_col, (size_t)nnz_local + 8);
    rc |= dev_alloc(&A->d_val, (size_t)nnz_local + 8);
    if (rc) {
        free_matrix_storage(A);
        delete A;
        return 1;
    }
    const int blocks = c->sm_count * 8;
    if (wide)
        hpcg_fill_kernel<int64_t><<<blocks, HPCG_FILL_ROWS, 0, c->stream>>>(rb, n_local, nx, ny, nz,
                                                                static_cast<int64_t *>(A->d_rp), A->d_col, A->d_val);
    else
        hpcg_fill_kernel<int32_t><<<blocks, HPCG_FILL_ROWS, 0, c->stream>>>(rb, n_local, nx, ny, nz,
                                                                static_cast<int32_t *>(A->d_rp), A->d_col, A->d_val);
    BIS_LAUNCH_CHECK(c);
    return finish_generated(c, A, out);
}

extern "C" int bis_matrix_generate_anderson(bis_context *c, int lx, int ly, int lz, double ranpot,
                                            double t, uint64_t seed, int periodic, bis_matrix **out) {
    BIS_REQUIRE(c && out, "null argument");
    BIS_REQUIRE(lx >= 1 && ly >= 1 && lz >= 1, "bis_matrix_generate_anderson: bad lattice");
    const int64_t n = (int64_t)lx * ly * lz;
    // row_ptr is 64-bit and the fill kernels index in 64 bits: only the column ids limit the lattice
    BIS_REQUIRE(n < INT32_MAX, "bis_matrix_generate_anderson: %lld sites exceed 32-bit column ids", (long long)n);
    BIS_CUDA(cudaSetDevice(c->device));
    bis_vector_cache_trim(c);
    int64_t rb = 0, re = n;
    slab(n, c->rank, c->nranks, (int64_t)lx * ly, &rb, &re);
    const int64_t n_local = re - rb;
    AndersonP p{lx, ly, lz, ranpot, t, seed, periodic};
    int64_t *d_rp64 = nullptr;
    BIS_CHECK(dev_alloc(&d_rp64, (size_t)n_local + 1 + 8));
    const int blocks = c->sm_count * 8;
    anderson_count_kernel<<<blocks, 256, 0, c->stream>>>(p, rb, n_local, d_rp64);
    BIS_LAUNCH_CHECK(c);
    thrust::exclusive_scan(thrust::cuda::par.on(c->stream), thrust::device_pointer_cast(d_rp64),
                           thrust::device_pointer_cast(d_rp64) + n_local + 1,
                           thrust::device_pointer_cast(d_rp64));
    int64_t nnz_local = 0;
    BIS_CUDA(cudaMemcpyAsync(&nnz_local, d_rp64 + n_local, sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    bis_matrix *A = new bis_matrix;
    A->n_rows = A->n_cols = n_local;
    A->n_rows_global = n;
    A->row_begin = rb;
    A->nnz = nnz_local;
    A->nnz_global = nnz_local;   // fixed below for nranks > 1
    A->max_row = 7;
    A->grid_nx = lx; A->grid_ny = ly; A->grid_nz = lz;
    A->mean_row = n_local ? (double)nnz_local / (double)n_local : 0.0;
    A->rp_bytes = 8;
    A->d_rp = d_rp64;
    if (dev_alloc(&A->d_col, (size_t)nnz_local + 8) || dev_alloc(&A->d_val, (size_t)nnz_local + 8)) {
        free_matrix_storage(A);
        delete A;
        return 1;
    }
    anderson_fill_kernel<<<blocks, 256, 0, c->stream>>>(p, rb, n_local, d_rp64, A->d_col, A->d_val);
    BIS_LAUNCH_CHECK(c);
    return finish_generated(c, A, out);
}

extern "C" int bis_matrix_free(bis_context *c, bis_matrix *A) {
    if (!A) return 0;
    if (c) {
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->stream);
        cudaStreamSynchronize(c->comm_stream);
    }
    free_matrix_storage(A);
    delete A;
    return 0;
}

extern "C" int bis_matrix_info(const bis_matrix *A, int64_t info[8]) {
    BIS_REQUIRE(A && info, "null argument");
    info[0] = A->n_rows;
    info[1] = A->n_rows_global;
    info[2] = A->nnz;
    info[3] = A->nnz_global;
    info[4] = A->rp_bytes;
    info[5] = A->lv.n_levels;
    info[6] = A->halo.n_ghost;
    info[7] = A->row_begin;
    return 0;
}

namespace {
__global__ void cols_to_global_kernel(int64_t nnz, const int *col, int64_t n_owned, int64_t row_begin,
                                      const int *ghost_global, int *out) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nnz;
         k += (int64_t)gridDim.x * blockDim.x) {
        int cc = col[k];
        out[k] = cc < n_owned ? (int)(cc + row_begin) : ghost_global[cc - n_owned];
    }
}
template <typename RP> __global__ void rp_to_i64_kernel(int64_t n1, const RP *rp, int64_t *out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n1;
         i += (int64_t)gridDim.x * blockDim.x)
        out[i] = (int64_t)rp[i];
}
} // namespace

extern "C" int bis_matrix_download_crs(bis_context *c, const bis_matrix *A, int64_t *rp, int32_t *col,
                                       double *val) {
    BIS_REQUIRE(c && A && rp, "null argument");
    BIS_REQUIRE_CRS(A);
    BIS_CUDA(cudaSetDevice(c->device));
    int64_t *d_rp64 = nullptr;
    BIS_CHECK(dev_alloc(&d_rp64, (size_t)A->n_rows + 1));
    if (A->rp_bytes == 8)
        rp_to_i64_kernel<int64_t><<<256, 256, 0, c->stream>>>(A->n_rows + 1, static_cast<const int64_t *>(A->d_rp), d_rp64);
    else
        rp_to_i64_kernel<int32_t><<<256, 256, 0, c->stream>>>(A->n_rows + 1, static_cast<const int32_t *>(A->d_rp), d_rp64);
    BIS_LAUNCH_CHECK(c);
    BIS_CUDA(cudaMemcpyAsync(rp, d_rp64, sizeof(int64_t) * ((size_t)A->n_rows + 1), cudaMemcpyDeviceToHost, c->stream));
    if (A->nnz && col) {
        int *d_tmp = nullptr;
        BIS_CHECK(dev_alloc(&d_tmp, (size_t)A->nnz));
        cols_to_global_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(A->nnz, A->d_col, A->n_cols, A->row_begin,
                                                                    A->halo.d_ghost_global, d_tmp);
        BIS_LAUNCH_CHECK(c);
        BIS_CUDA(cudaMemcpyAsync(col, d_tmp, sizeof(int32_t) * (size_t)A->nnz, cudaMemcpyDeviceToHost, c->stream));
        BIS_CUDA(cudaStreamSynchronize(c->stream));
        cudaFree(d_tmp);
    }
    if (A->nnz && val)
        BIS_CUDA(cudaMemcpyAsync(val, A->d_val, sizeof(double) * (size_t)A->nnz, cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(d_rp64);
    return 0;
}

namespace {
template <typename RP>
__global__ void extract_diag_kernel(int64_t n, const RP *rp, const int *col, const double *val,
                                    double *D, double *D_inv, int *missing) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n;
         r += (int64_t)gridDim.x * blockDim.x) {
        bool found = false;
        for (RP k = rp[r]; k < rp[r + 1]; ++k) {
            if (col[k] == r) {   // local column id == local row id on the diagonal
                double d = val[k];
                D[r] = d;
                if (fabs(d) < 1e-16)   // SanityChecker::zero_diag (LU_factors.hpp:842-845)
                    atomicExch(missing + 1, (int)(r + 1 > 0x7fffffff ? 0x7fffffff : r + 1));
                if (D_inv) D_inv[r] = div_rn(1.0, d);
                found = true;   // peel_diag_crs_new keeps the LAST match (LU_factors.hpp:836-850)
            }
        }
        if (!found) atomicExch(missing, (int)(r + 1 > 0x7fffffff ? 0x7fffffff : r + 1));
    }
}
} // namespace

extern "C" int bis_matrix_extract_diagonal(bis_context *c, const bis_matrix *A, double *D, double *D_inv) {
    BIS_REQUIRE(c && A && D, "null argument");
    BIS_REQUIRE_CRS(A);
    BIS_CUDA(cudaSetDevice(c->device));
    int *d_missing = nullptr;
    BIS_CHECK(dev_alloc(&d_missing, 2));
    BIS_CUDA(cudaMemsetAsync(d_missing, 0, 2 * sizeof(int), c->stream));
    const int blocks = bis_blocks_for(A->n_rows, 256, c->sm_count * 8);
    if (A->rp_bytes == 8)
        extract_diag_kernel<int64_t><<<blocks, 256, 0, c->stream>>>(A->n_rows, static_cast<const int64_t *>(A->d_rp), A->d_col, A->d_val, D, D_inv, d_missing);
    else
        extract_diag_kernel<int32_t><<<blocks, 256, 0, c->stream>>>(A->n_rows, static_cast<const int32_t *>(A->d_rp), A->d_col, A->d_val, D, D_inv, d_missing);
    BIS_LAUNCH_CHECK(c);
    int missing[2] = {0, 0};
    BIS_CUDA(cudaMemcpyAsync(missing, d_missing, 2 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(d_missing);
    // SanityChecker::no_diag / zero_diag (common.hpp:388-396) are fatal in the reference
    BIS_REQUIRE(missing[0] == 0, "No diagonal to extract at row index %d", missing[0] - 1);
    BIS_REQUIRE(missing[1] == 0, "Zero detected on diagonal at row index %d", missing[1] - 1);
    return 0;
}

// ---- -scale: symmetric diagonal scaling (preprocessing.hpp:8-24,39-50, LU_factors.hpp:880-898) ----
namespace {
template <typename RP>
__global__ void scale_extract_kernel(int64_t n, const RP *rp, const int *col, const double *val, double *s, int *zero) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
        double sr = 0.0;   // A_D_scale starts at 0.0 (solver.hpp:105) and keeps it for a row without diagonal
        for (RP k = rp[r]; k < rp[r + 1]; ++k)
            if (col[k] == r) {
                const double d = val[k];
                if (fabs(d) < 1e-16) atomicExch(zero, (int)(r + 1 > 0x7fffffff ? 0x7fffffff : r + 1));
                sr = div_rn(1.0, sqrt(fabs(d)));
            }
        s[r] = sr;
    }
}
template <typename RP>
__global__ void scale_apply_kernel(int64_t n, const RP *rp, const int *col, double *val, const double *s,
                                   const double *ghost, int64_t n_owned) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
        const double sr = s[r];
        for (RP k = rp[r]; k < rp[r + 1]; ++k) {
            const int c = col[k];
            const double sc = c < n_owned ? s[c] : ghost[c - n_owned];
            val[k] = mul_rn(val[k], mul_rn(sr, sc));   // A->val[i] *= (s_row * s_col)
        }
    }
}
} // namespace

extern "C" int bis_matrix_scale_symmetric(bis_context *c, bis_matrix *A, double *D_scale) {
    BIS_REQUIRE(c && A && D_scale, "null argument");
    BIS_REQUIRE_CRS(A);
    BIS_REQUIRE(A->triangular == 0, "bis_matrix_scale_symmetric: general matrices only");
    BIS_CUDA(cudaSetDevice(c->device));
    const int64_t n = A->n_rows;
    int *d_zero = nullptr;
    BIS_CHECK(dev_alloc(&d_zero, 1));
    BIS_CUDA(cudaMemsetAsync(d_zero, 0, sizeof(int), c->stream));
    const int blocks = bis_blocks_for(n, 256, c->sm_count * 8);
    if (A->rp_bytes == 8)
        scale_extract_kernel<int64_t><<<blocks, 256, 0, c->stream>>>(n, static_cast<const int64_t *>(A->d_rp), A->d_col, A->d_val, D_scale, d_zero);
    else
        scale_extract_kernel<int32_t><<<blocks, 256, 0, c->stream>>>(n, static_cast<const int32_t *>(A->d_rp), A->d_col, A->d_val, D_scale, d_zero);
    BIS_LAUNCH_CHECK(c);
    int zero = 0;
    BIS_CUDA(cudaMemcpyAsync(&zero, d_zero, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(d_zero);
    BIS_REQUIRE(zero == 0, "Zero detected on diagonal at row index %d", zero - 1);
    // the column factors of ghost columns come from their owners
    if (A->distributed) {
        BIS_CHECK(bis_halo_exchange_begin(c, A, D_scale));
        BIS_CHECK(bis_halo_exchange_end(c, A));
    }
    if (A->rp_bytes == 8)
        scale_apply_kernel<int64_t><<<blocks, 256, 0, c->stream>>>(n, static_cast<const int64_t *>(A->d_rp), A->d_col, A->d_val, D_scale, A->halo.cur_ghost, A->n_cols);
    else
        scale_apply_kernel<int32_t><<<blocks, 256, 0, c->stream>>>(n, static_cast<const int32_t *>(A->d_rp), A->d_col, A->d_val, D_scale, A->halo.cur_ghost, A->n_cols);
    BIS_LAUNCH_CHECK(c);
    bis_win_values_changed(A);
    return 0;
}
