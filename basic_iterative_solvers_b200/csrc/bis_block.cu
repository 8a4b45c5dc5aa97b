// bis_block.cu -- several right-hand sides against one matrix (include/bis_b200.h, "multiple right-hand
// sides"): the CRS SpMM Y = A X and the streaming kernels of a block CG whose every column is, bit for bit,
// the single-vector composition bis_spmv / bis_dot_to_slot / bis_cg_update / bis_cg_direction_x.
//
// Layout: a block of k vectors is an n x k ROW-MAJOR array, element (i, j) at V[i*k + j] (one gather of row
// `col` of X fetches k contiguous doubles).  Column j's scalars live in slots slot0 + j.
//
// SpMM bit rule: Y[i, j] is native_spmv on column j -- products val*x rounded separately, added left to right
// in storage order starting from 0.0 -- so each column equals oracle/port.spmv for every matrix, and bis_spmv
// whenever that takes the TMA-tile or the windowed variant.
//
// Streaming reduction rule: the rows of a block, and the order in which a thread adds its rows into a column's
// accumulator, are those of ew_kernel (bis_blas1.cu): block b owns rows [b*chunk, (b+1)*chunk), 256 threads,
// thread t adds rows t, t+256, t+512, t+768 of each 1024-row trip in that order with fma, then the same warp
// and block shuffle trees, the same per-slab sums and combine_records.  Only the loads differ (a thread reads
// the k contiguous values of its row).
#include "bis_device.cuh"
#include "bis_spmv_tma.cuh"

#include <cfloat>
#include <cstring>

namespace {

constexpr int KMAX = BIS_BLOCK_MAX_K;
constexpr int BW_THREADS = 256;     // == EW_THREADS of bis_blas1.cu
constexpr int BW_UNROLL = 4;        // == EW_UNROLL
constexpr int BQ_MAX = 2 * KMAX;    // reduced quantities per launch

// ---- SpMM ----------------------------------------------------------------------------------------------
// A tile of R consecutive rows is staged by two TMA bulk copies (val[], col[]) as in SpMV variant 2
// (bis_spmv_tma.cuh); a row is served by TPR threads, each owning CW consecutive columns of the block and one
// accumulator per column, walking the row's nonzeros in storage order.  The TPR threads of a row gather
// neighbouring 16-byte pieces of the same X row (K = 16: one 128-byte line per row and nonzero).
template <int K> struct SpmmShape {
    static constexpr int TPR = K <= 4 ? 1 : (K <= 8 ? 2 : 4);               // threads per row
    static constexpr bool VEC = (K % 2) == 0;                               // 16-byte gathers and stores
    static constexpr int CW = VEC ? 2 * ((K + 2 * TPR - 1) / (2 * TPR)) : (K + TPR - 1) / TPR;   // columns per thread
    static constexpr int U = CW <= 2 ? 8 : 4;                               // nonzeros whose gathers are in flight together
};

struct SpmmIn {
    const void *rp;
    const int *col;
    const double *val;
    const double *X;
    double *Y;
    int64_t n_rows;
    int cap;
    int nstage;
    int rows;   // rows per tile
};

// acc[w] += val * X[c, c0 + w] for the columns this thread owns (w < ncw), one product at a time
template <int K>
__device__ __forceinline__ void spmm_gather(const double *__restrict__ X, int c, int c0, double (&xv)[SpmmShape<K>::CW]) {
    using S = SpmmShape<K>;
    const double *p = X + (int64_t)c * K + c0;
    if constexpr (S::VEC) {
#pragma unroll
        for (int w = 0; w < S::CW; w += 2) {
            if (c0 + w < K) {
                const double2 t = __ldg(reinterpret_cast<const double2 *>(p + w));
                xv[w] = t.x;
                xv[w + 1] = t.y;
            } else {
                xv[w] = xv[w + 1] = 0.0;
            }
        }
    } else {
#pragma unroll
        for (int w = 0; w < S::CW; ++w) xv[w] = (c0 + w < K) ? __ldg(p + w) : 0.0;
    }
}

template <int K>
__device__ __forceinline__ void spmm_store(double *__restrict__ Y, int64_t row, int c0, const double (&acc)[SpmmShape<K>::CW]) {
    using S = SpmmShape<K>;
    double *p = Y + row * K + c0;
    if constexpr (S::VEC) {
#pragma unroll
        for (int w = 0; w < S::CW; w += 2)
            if (c0 + w < K) *reinterpret_cast<double2 *>(p + w) = make_double2(acc[w], acc[w + 1]);
    } else {
#pragma unroll
        for (int w = 0; w < S::CW; ++w)
            if (c0 + w < K) p[w] = acc[w];
    }
}

// one row, nonzeros [a, b) of (col, val), in storage order
template <int K, class ColF, class ValF>
__device__ __forceinline__ void spmm_row(const double *__restrict__ X, int64_t a, int64_t b, int c0, ColF colf, ValF valf,
                                         double (&acc)[SpmmShape<K>::CW]) {
    using S = SpmmShape<K>;
#pragma unroll
    for (int w = 0; w < S::CW; ++w) acc[w] = 0.0;
    int64_t k = a;
    for (; k + S::U <= b; k += S::U) {
        int c[S::U];
        double v[S::U];
        double xv[S::U][S::CW];
#pragma unroll
        for (int u = 0; u < S::U; ++u) {
            c[u] = colf(k + u);
            v[u] = valf(k + u);
        }
#pragma unroll
        for (int u = 0; u < S::U; ++u) spmm_gather<K>(X, c[u], c0, xv[u]);
#pragma unroll
        for (int u = 0; u < S::U; ++u)
#pragma unroll
            for (int w = 0; w < S::CW; ++w) acc[w] = add_rn(acc[w], mul_rn(v[u], xv[u][w]));
    }
    for (; k < b; ++k) {
        double xv[S::CW];
        const double v = valf(k);
        spmm_gather<K>(X, colf(k), c0, xv);
#pragma unroll
        for (int w = 0; w < S::CW; ++w) acc[w] = add_rn(acc[w], mul_rn(v, xv[w]));
    }
}

template <typename RP, int K>
__global__ void __launch_bounds__(512, 1) spmm_tma_kernel(SpmmIn in) {
    using S = SpmmShape<K>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw);                       // [MAX_STAGES]
    double *sval = reinterpret_cast<double *>(smem_raw + 128);                     // [nstage][cap]
    int *scol = reinterpret_cast<int *>(smem_raw + 128 + (size_t)in.nstage * in.cap * sizeof(double));

    const RP *__restrict__ rp = static_cast<const RP *>(in.rp);
    const int R = in.rows;
    const int64_t n_tiles = (in.n_rows + R - 1) / R;
    // interleaved static tile -> CTA map (as SpMV variant 2): all CTAs sweep the matrix together
    const int64_t t_first = blockIdx.x, t_stride = gridDim.x;
    const int64_t my_tiles = n_tiles > t_first ? (n_tiles - t_first + t_stride - 1) / t_stride : 0;
    const int rl = (int)threadIdx.x / S::TPR;
    const int c0 = ((int)threadIdx.x % S::TPR) * S::CW;

    if (threadIdx.x == 0) {
        for (int s = 0; s < in.nstage; ++s) tma::mbar_init(&bars[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    uint64_t policy = 0;
    if (threadIdx.x == 0) policy = tma::policy_evict_first();

    auto tile_range = [&](int64_t j, int64_t &s, int64_t &e) {
        if (j >= my_tiles) {
            s = e = 0;
            return;
        }
        const int64_t r0 = (t_first + j * t_stride) * R;
        int64_t r1 = r0 + R;
        if (r1 > in.n_rows) r1 = in.n_rows;
        s = (int64_t)rp[r0];
        e = (int64_t)rp[r1];
    };
    auto issue = [&](int64_t j, int64_t s, int64_t e) {
        const int64_t s_al = s & ~(int64_t)3;
        const int64_t e_al = (e + 3) & ~(int64_t)3;
        const uint32_t n_el = (uint32_t)(e_al - s_al);
        const int st = (int)(j % in.nstage);
        if (n_el == 0) {
            tma::mbar_arrive(&bars[st]);
            return;
        }
        tma::fence_reads_before_bulk_write();
        tma::mbar_expect_tx(&bars[st], n_el * 12u);
        tma::bulk_g2s(sval + (size_t)st * in.cap, in.val + s_al, n_el * 8u, &bars[st], policy);
        tma::bulk_g2s(scol + (size_t)st * in.cap, in.col + s_al, n_el * 4u, &bars[st], policy);
    };
    if (threadIdx.x == 0) {
        const int64_t pre = my_tiles < in.nstage ? my_tiles : in.nstage;
        for (int64_t j = 0; j < pre; ++j) {
            int64_t s, e;
            tile_range(j, s, e);
            issue(j, s, e);
        }
    }
    auto row_bounds = [&](int64_t j, int64_t &ks, int64_t &ke, int64_t &row) {
        row = (t_first + j * t_stride) * R + rl;
        if (j < my_tiles && row < in.n_rows && c0 < K) {
            ks = (int64_t)rp[row];
            ke = (int64_t)rp[row + 1];
        } else {
            ks = ke = 0;
            row = -1;
        }
    };
    int64_t ts, te, ks, ke, row;
    tile_range(0, ts, te);
    row_bounds(0, ks, ke, row);
    for (int64_t j = 0; j < my_tiles; ++j) {
        const int st = (int)(j % in.nstage);
        const uint32_t parity = (uint32_t)((j / in.nstage) & 1);
        int64_t nts, nte, nks, nke, nrow, is = 0, ie = 0;
        tile_range(j + 1, nts, nte);
        row_bounds(j + 1, nks, nke, nrow);
        if (threadIdx.x == 0) tile_range(j + in.nstage, is, ie);
        tma::mbar_wait(&bars[st], parity);
        if (row >= 0) {
            const int64_t base = ts & ~(int64_t)3;
            const double *__restrict__ sv = sval + (size_t)st * in.cap;
            const int *__restrict__ sc = scol + (size_t)st * in.cap;
            double acc[S::CW];
            spmm_row<K>(in.X, ks - base, ke - base, c0, [&](int64_t k) { return sc[k]; },
                        [&](int64_t k) { return sv[k]; }, acc);
            spmm_store<K>(in.Y, row, c0, acc);
        }
        __syncthreads();   // every thread is done with stage `st`
        if (threadIdx.x == 0 && j + in.nstage < my_tiles) issue(j + in.nstage, is, ie);
        ts = nts; te = nte; ks = nks; ke = nke; row = nrow;
    }
}

// Rows too long for a shared-memory tile: the same per-thread walk straight from global memory.
template <typename RP, int K>
__global__ void __launch_bounds__(256) spmm_direct_kernel(SpmmIn in) {
    using S = SpmmShape<K>;
    const RP *__restrict__ rp = static_cast<const RP *>(in.rp);
    const int *__restrict__ col = in.col;
    const double *__restrict__ val = in.val;
    const int c0 = ((int)threadIdx.x % S::TPR) * S::CW;
    if (c0 >= K) return;
    const int64_t stride = (int64_t)gridDim.x * (blockDim.x / S::TPR);
    for (int64_t row = (int64_t)blockIdx.x * (blockDim.x / S::TPR) + threadIdx.x / S::TPR; row < in.n_rows; row += stride) {
        double acc[S::CW];
        spmm_row<K>(in.X, (int64_t)rp[row], (int64_t)rp[row + 1], c0, [&](int64_t k) { return ld_stream(col + k); },
                    [&](int64_t k) { return ld_stream(val + k); }, acc);
        spmm_store<K>(in.Y, row, c0, acc);
    }
}

bool spmm_plan(const bis_matrix *A, int tpr, int *rows, int *cap, size_t *smem) {
    const size_t budget = (size_t)110 << 10;   // two stages; two CTAs per SM where registers allow
    for (int R : {256, 128, 64, 32}) {
        if (R * tpr > 512) continue;
        const int c = (int)(((int64_t)R * A->max_row + 8 + 3) & ~(int64_t)3);
        const size_t stage = (size_t)c * 12;
        if (128 + 2 * stage > budget && R > 32) continue;
        if (128 + 2 * stage > ((size_t)220 << 10)) return false;
        *rows = R;
        *cap = c;
        *smem = 128 + 2 * stage;
        return true;
    }
    return false;
}

template <typename RP, int K>
int launch_spmm(bis_context *c, const bis_matrix *A, const double *X, double *Y) {
    using S = SpmmShape<K>;
    SpmmIn in;
    in.rp = A->d_rp; in.col = A->d_col; in.val = A->d_val; in.X = X; in.Y = Y; in.n_rows = A->n_rows;
    in.cap = 0; in.nstage = 2; in.rows = 0;
    int R = 0, cap = 0;
    size_t smem = 0;
    if (A->max_row >= 1 && spmm_plan(A, S::TPR, &R, &cap, &smem)) {
        auto kern = spmm_tma_kernel<RP, K>;
        BIS_CHECK(bis_ensure_dynamic_smem(c, reinterpret_cast<const void *>(kern), smem));
        const int threads = R * S::TPR;
        int occ = 1;
        BIS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
        if (occ < 1) occ = 1;
        const int64_t n_tiles = (A->n_rows + R - 1) / R;
        int64_t grid = (int64_t)c->sm_count * occ;
        if (grid > n_tiles) grid = n_tiles;
        if (grid < 1) grid = 1;
        in.cap = cap;
        in.rows = R;
        kern<<<(unsigned)grid, threads, smem, c->stream>>>(in);
    } else {
        const int rows_per_block = 256 / S::TPR;
        const int blocks = bis_blocks_for(A->n_rows, rows_per_block, c->sm_count * 8);
        spmm_direct_kernel<RP, K><<<blocks, 256, 0, c->stream>>>(in);
    }
    BIS_LAUNCH_CHECK(c);
    return 0;
}

// ---- batched streaming kernels -------------------------------------------------------------------------
enum BlockOp { OP_DOT = 0, OP_RESID = 1, OP_UPDATE = 2, OP_DIRX = 3 };

template <int K, int OP> struct BlockNq {
    static constexpr int value = OP == OP_DOT ? K : (OP == OP_DIRX ? 0 : 2 * K);
};

struct BlockArgs {
    int64_t n;
    int chunk;
    int jacobi;
    const double *in0, *in1, *in2;   // per OP, see the kernel
    const double *D;                 // [n] diagonal (Jacobi)
    double *out0, *out1, *out2;
    const double *S;                 // device scalars
    int slot_a, slot_b, slot_c;      // scalar slot ranges read by the prologue
    const double *state;             // [3k] block-CG state (thresholds, active flags, iterations) or NULL: all active
    double *partials;                // [2*KMAX][BIS_MAX_RED_BLOCKS]
    int slot_q[BQ_MAX];              // target slot of every reduced quantity (-1: not written)
};

// Sum of NQ quantities over the grid.  Every step is that of block_reduce_finish / grid_reduce_finish (bis_device.cuh)
// on one GPU -- the same shuffle trees over the same numbers, the same per-slab order, combine_records over the
// n_rec records -- only spread over the warps of the block differently.  Quantity q belongs to column q % K;
// the slot of an inactive column is not written.
template <int K, int NQ>
__device__ __forceinline__ void block_reduce_multi(double (&acc)[NQ > 0 ? NQ : 1], const BlockArgs &a, const RedArgs &ra,
                                                   const bool *s_act) {
    __shared__ double s_part[NQ][32];
    __shared__ double s_rec[NQ][BIS_NSLAB];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int nwarp = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
        const double v = warp_sum(acc[q]);
        if (lane == 0) s_part[q][warp] = v;
    }
    __syncthreads();
    for (int q = warp; q < NQ; q += nwarp) {
        double v = (lane < nwarp) ? s_part[q][lane] : 0.0;
        v = warp_sum(v);
        if (lane == 0) {
            a.partials[q * BIS_MAX_RED_BLOCKS + blockIdx.x] = v;
            __threadfence();
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned int ticket = atomicAdd(ra.counter, 1u);
        s_last = (ticket == gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int w = warp; w < ra.n_slab * NQ; w += nwarp) {
        const int i = w / NQ, q = w % NQ;
        const int lo = ra.slab_off[i], hi = ra.slab_off[i + 1];
        const double *p = a.partials + q * BIS_MAX_RED_BLOCKS;
        double v = 0.0;
        int j = lo + lane;
        for (; j + 7 * 32 < hi; j += 8 * 32) {
            double t[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) t[u] = __ldcg(p + j + u * 32);
#pragma unroll
            for (int u = 0; u < 8; ++u) v += t[u];
        }
        for (; j < hi; j += 32) v += __ldcg(p + j);
        v = warp_sum(v);
        if (lane == 0) s_rec[q][i] = v;
    }
    __syncthreads();
    if ((int)threadIdx.x < NQ) {
        const int q = threadIdx.x;
        double r[BIS_NSLAB];
#pragma unroll
        for (int i = 0; i < BIS_NSLAB; ++i) r[i] = i < ra.n_rec ? s_rec[q][i] : 0.0;
        // combine_records with its loop unrolled (no local-memory array)
        double t;
        if (ra.n_rec == BIS_NSLAB) {
            t = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
        } else {
            t = 0.0;
#pragma unroll
            for (int i = 0; i < BIS_NSLAB; ++i)
                if (i < ra.n_rec) t += r[i];
        }
        if (a.slot_q[q] >= 0 && s_act[q % K]) ra.scalars[a.slot_q[q]] = t;
    }
    __syncthreads();
    if (threadIdx.x == 0) *ra.counter = 0u;
}

// One element (row i, column j) of each operation, with the arithmetic of the single-vector kernel it batches.
//  OP_DOT    in0 = A, in1 = B                          acc[j] += a*b                      (bis_dot_to_slot)
//  OP_RESID  in0 = AX, in1 = B -> out0 = R, out1 = Z, out2 = P (optional)
//            r = B - AX (bis_subtract_vectors, scale 1); z = r / (1.0*D) (bis_elemwise_div_vectors) or r;
//            acc[j] += r*z (bis_dot_to_slot), acc[K+j] += r*r (bis_sumsq_to_slot)
//  OP_UPDATE in0 = R_old, in1 = AP -> out0 = R_new, out1 = Z_new                        (bis_cg_update, x_new NULL)
//            acc[j] += r*r, acc[K+j] += r*z
//  OP_DIRX   in0 = Z_new, in1 = P_old, in2 = X_old -> out0 = P_new, out1 = X_new       (bis_cg_direction_x)
//            a column that is not active carries X_old into X_new and leaves P_new alone
template <int K, int OP>
__global__ void __launch_bounds__(BW_THREADS, 1) block_ew_kernel(BlockArgs a, RedArgs ra) {
    constexpr int NQ = BlockNq<K, OP>::value;
    __shared__ double s_c0[K], s_c1[K];
    __shared__ bool s_act[K];
    if ((int)threadIdx.x < K) {
        const int j = threadIdx.x;
        s_act[j] = a.state == nullptr || a.state[K + j] != 0.0;
        if (OP == OP_UPDATE) s_c0[j] = div_rn(a.S[a.slot_a + j], a.S[a.slot_b + j]);            // alpha = rz / pAp
        if (OP == OP_DIRX) {
            s_c0[j] = div_rn(a.S[a.slot_b + j], a.S[a.slot_c + j]);                            // alpha = rz / pAp
            s_c1[j] = div_rn(a.S[a.slot_a + j], a.S[a.slot_b + j]);                            // beta = rz_new / rz
        }
    }
    __syncthreads();
    double acc[NQ > 0 ? NQ : 1];
#pragma unroll
    for (int q = 0; q < (NQ > 0 ? NQ : 1); ++q) acc[q] = 0.0;

    const int64_t base = (int64_t)blockIdx.x * a.chunk;
    const int64_t end = base + a.chunk < a.n ? base + a.chunk : a.n;
    constexpr int TRIP = BW_THREADS * BW_UNROLL;
    for (int64_t t0 = base; t0 < end; t0 += TRIP) {
#pragma unroll 1
        for (int u = 0; u < BW_UNROLL; ++u) {
            const int64_t i = t0 + threadIdx.x + u * BW_THREADS;
            if (i >= end) break;
            const int64_t o = i * K;
            if constexpr (OP == OP_DOT) {
                double x[K], y[K];
#pragma unroll
                for (int j = 0; j < K; ++j) { x[j] = a.in0[o + j]; y[j] = a.in1[o + j]; }
#pragma unroll
                for (int j = 0; j < K; ++j) acc[j] = fma(x[j], y[j], acc[j]);
            } else if constexpr (OP == OP_RESID) {
                double ax[K], b[K];
#pragma unroll
                for (int j = 0; j < K; ++j) { ax[j] = a.in0[o + j]; b[j] = a.in1[o + j]; }
                const double d = a.jacobi ? a.D[i] : 1.0;
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    const double r = fma(-1.0, ax[j], b[j]);
                    const double z = a.jacobi ? div_rn(r, mul_rn(1.0, d)) : r;
                    a.out0[o + j] = r;
                    a.out1[o + j] = z;
                    if (a.out2) a.out2[o + j] = z;
                    acc[j] = fma(r, z, acc[j]);
                    acc[K + j] = fma(r, r, acc[K + j]);
                }
            } else if constexpr (OP == OP_UPDATE) {
                double ro[K], ap[K];
#pragma unroll
                for (int j = 0; j < K; ++j) { ro[j] = a.in0[o + j]; ap[j] = a.in1[o + j]; }
                const double d = a.jacobi ? a.D[i] : 1.0;
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    const double r = fma(-s_c0[j], ap[j], ro[j]);
                    const double z = a.jacobi ? div_rn(r, d) : r;
                    if (s_act[j]) {
                        a.out0[o + j] = r;
                        a.out1[o + j] = z;
                    }
                    acc[j] = fma(r, r, acc[j]);
                    acc[K + j] = fma(r, z, acc[K + j]);
                }
            } else {
                double z[K], p[K], x[K];
#pragma unroll
                for (int j = 0; j < K; ++j) { z[j] = a.in0[o + j]; p[j] = a.in1[o + j]; x[j] = a.in2[o + j]; }
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    if (s_act[j]) {
                        a.out1[o + j] = fma(s_c0[j], p[j], x[j]);
                        a.out0[o + j] = fma(s_c1[j], p[j], z[j]);
                    } else {
                        a.out1[o + j] = x[j];
                    }
                }
            }
        }
    }
    if constexpr (NQ > 0) block_reduce_multi<K, NQ>(acc, a, ra, s_act);
}

// Device-side stop rule of a block CG (check_stopping_criteria, host/solver.hpp), latched once at the start of
// an iteration.  state: [0,k) stop thresholds tol*||r0_j||, [k,2k) active flags, [2k,3k) iterations done.
__global__ void block_cg_status_kernel(int k, const double *S, int slot_rr, int max_iters, double *state) {
    const int j = threadIdx.x;
    if (j >= k || state[k + j] == 0.0) return;
    const double it = state[2 * k + j];
    bool active = true;
    if (it > 0.0) {
        const double nrm = sqrt(S[slot_rr + j]);
        if (fabs(nrm) < state[j] || fabs(nrm) > DBL_MAX || isnan(nrm)) active = false;
    }
    if (active && it >= (double)max_iters) active = false;
    if (active) state[2 * k + j] = it + 1.0;
    else state[k + j] = 0.0;
}

int ensure_block_partials(bis_context *c) {
    if (c->d_block_partials) return 0;
    BIS_REQUIRE(!c->capturing, "multi-RHS kernels: the first reducing call must not be recorded into a graph");
    BIS_CUDA(bis_cuda_malloc(&c->d_block_partials, sizeof(double) * BQ_MAX * BIS_MAX_RED_BLOCKS));
    return 0;
}

template <int K, int OP>
int launch_block_k(bis_context *c, BlockArgs a) {
    constexpr int NQ = BlockNq<K, OP>::value;
    RedArgs ra = bis_red_args(c, -1, -1);
    int64_t blocks;
    const int64_t n = a.n;
    if (NQ > 0) {
        // the launch shape and slab layout of launch_ew2 (bis_blas1.cu) for a reducing kernel over n rows
        BIS_CHECK(ensure_block_partials(c));
        const RowPartition part = bis_partition_for(c, n);
        int chunk = part.chunk;
        while ((n + chunk - 1) / chunk > BIS_MAX_RED_BLOCKS) chunk <<= 1;
        blocks = (n + chunk - 1) / chunk;
        int off[BIS_NSLAB + 1];
        bool aligned = chunk == part.chunk;
        for (int i = 0; i <= part.n_slab; ++i) {
            off[i] = (int)((part.slab_row[i] + chunk - 1) / chunk);
            if (i < part.n_slab && part.slab_row[i] % chunk != 0) aligned = false;
        }
        RowPartition eff = part;
        if (!aligned) eff.invariant = false;
        bis_red_set_slabs(c, ra, eff, off, (int)(blocks > 0 ? blocks : 1));
        a.chunk = chunk;
        a.partials = c->d_block_partials;
    } else {
        a.chunk = 4096;
        blocks = (n + a.chunk - 1) / a.chunk;
    }
    if (blocks < 1) blocks = 1;
    BIS_CHECK(bis_prof_begin(c, BIS_PROF_VECTOR));
    block_ew_kernel<K, OP><<<(unsigned)blocks, BW_THREADS, 0, c->stream>>>(a, ra);
    BIS_LAUNCH_CHECK(c);
    BIS_CHECK(bis_prof_end(c, BIS_PROF_VECTOR));
    return 0;
}

template <int OP>
int launch_block(bis_context *c, int k, const BlockArgs &a) {
    switch (k) {
#define BIS_BLOCK_CASE(K) case K: return launch_block_k<K, OP>(c, a);
    BIS_BLOCK_CASE(1) BIS_BLOCK_CASE(2) BIS_BLOCK_CASE(3) BIS_BLOCK_CASE(4) BIS_BLOCK_CASE(5) BIS_BLOCK_CASE(6)
    BIS_BLOCK_CASE(7) BIS_BLOCK_CASE(8) BIS_BLOCK_CASE(9) BIS_BLOCK_CASE(10) BIS_BLOCK_CASE(11) BIS_BLOCK_CASE(12)
    BIS_BLOCK_CASE(13) BIS_BLOCK_CASE(14) BIS_BLOCK_CASE(15) BIS_BLOCK_CASE(16)
#undef BIS_BLOCK_CASE
    }
    bis_set_error("multi-RHS: k = %d outside [1, %d]", k, KMAX);
    return 2;
}

template <typename RP>
int launch_spmm_rp(bis_context *c, const bis_matrix *A, int k, const double *X, double *Y) {
    switch (k) {
#define BIS_SPMM_CASE(K) case K: return launch_spmm<RP, K>(c, A, X, Y);
    BIS_SPMM_CASE(1) BIS_SPMM_CASE(2) BIS_SPMM_CASE(3) BIS_SPMM_CASE(4) BIS_SPMM_CASE(5) BIS_SPMM_CASE(6)
    BIS_SPMM_CASE(7) BIS_SPMM_CASE(8) BIS_SPMM_CASE(9) BIS_SPMM_CASE(10) BIS_SPMM_CASE(11) BIS_SPMM_CASE(12)
    BIS_SPMM_CASE(13) BIS_SPMM_CASE(14) BIS_SPMM_CASE(15) BIS_SPMM_CASE(16)
#undef BIS_SPMM_CASE
    }
    bis_set_error("bis_spmm: k = %d outside [1, %d]", k, KMAX);
    return 2;
}

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

BlockArgs block_args(bis_context *c, int64_t n) {
    BlockArgs a;
    memset(&a, 0, sizeof a);
    a.n = n;
    a.S = c->d_scalars;
    for (int q = 0; q < BQ_MAX; ++q) a.slot_q[q] = -1;
    return a;
}

} // namespace

// common checks of every multi-RHS entry point
#define REQ_BLOCK(c, k)                                                                                      \
    do {                                                                                                     \
        BIS_REQUIRE((c) != nullptr, "null context");                                                         \
        BIS_REQUIRE((c)->nranks == 1, "multi-RHS entry points are single-GPU only (distributed context)");  \
        BIS_REQUIRE((k) >= 1 && (k) <= KMAX, "multi-RHS: k = %d outside [1, %d]", (k), KMAX);               \
    } while (0)
#define REQ_BLOCK_VEC(p, what) BIS_REQUIRE((p) != nullptr && aligned16(p), "multi-RHS: %s is null or not 16-byte aligned", what)
#define REQ_SLOTS(s, k, what) \
    BIS_REQUIRE((s) >= 0 && (s) + (k) <= BIS_NUM_SCALARS, "multi-RHS: slots %s [%d, %d) outside [0, %d)", what, (s), (s) + (k), BIS_NUM_SCALARS)

extern "C" int bis_spmm(bis_context *c, const bis_matrix *A, int k, const double *X, double *Y) {
    REQ_BLOCK(c, k);
    BIS_REQUIRE(A, "bis_spmm: null matrix");
    BIS_REQUIRE(!A->distributed, "bis_spmm: distributed matrices are not supported");
    BIS_REQUIRE_CRS(A);
    REQ_BLOCK_VEC(X, "X");
    REQ_BLOCK_VEC(Y, "Y");
    BIS_REQUIRE(X != Y, "bis_spmm: X and Y must not alias");
    BisNvtxRange nvtx_range("spmm");
    BIS_CUDA(cudaSetDevice(c->device));
    BIS_CHECK(bis_prof_begin(c, BIS_PROF_SPMV));
    if (A->rp_bytes == 8) BIS_CHECK(launch_spmm_rp<int64_t>(c, A, k, X, Y));
    else BIS_CHECK(launch_spmm_rp<int32_t>(c, A, k, X, Y));
    BIS_CHECK(bis_prof_end(c, BIS_PROF_SPMV));
    return 0;
}

extern "C" int bis_block_dot_to_slots(bis_context *c, int64_t n, int k, const double *A, const double *B, int slot0,
                                      const double *state) {
    REQ_BLOCK(c, k);
    REQ_BLOCK_VEC(A, "A");
    REQ_BLOCK_VEC(B, "B");
    REQ_SLOTS(slot0, k, "slot0");
    BlockArgs a = block_args(c, n);
    a.in0 = A; a.in1 = B; a.state = state;
    for (int j = 0; j < k; ++j) a.slot_q[j] = slot0 + j;
    return launch_block<OP_DOT>(c, k, a);
}

extern "C" int bis_block_residual(bis_context *c, int precond, int64_t n, int k, const double *AX, const double *B,
                                  const double *A_D, double *R, double *Z, double *P, int slot_rz0, int slot_rr0) {
    REQ_BLOCK(c, k);
    BIS_REQUIRE(precond == BIS_PRECOND_NONE || precond == BIS_PRECOND_JACOBI,
                "bis_block_residual: preconditioner %d not supported (none or jacobi)", precond);
    REQ_BLOCK_VEC(AX, "AX"); REQ_BLOCK_VEC(B, "B"); REQ_BLOCK_VEC(R, "R"); REQ_BLOCK_VEC(Z, "Z");
    BIS_REQUIRE(P == nullptr || aligned16(P), "bis_block_residual: P not 16-byte aligned");
    BIS_REQUIRE(precond != BIS_PRECOND_JACOBI || A_D, "bis_block_residual: jacobi needs A_D");
    REQ_SLOTS(slot_rz0, k, "rz"); REQ_SLOTS(slot_rr0, k, "rr");
    BlockArgs a = block_args(c, n);
    a.jacobi = precond == BIS_PRECOND_JACOBI;
    a.in0 = AX; a.in1 = B; a.D = A_D; a.out0 = R; a.out1 = Z; a.out2 = P;
    for (int j = 0; j < k; ++j) {
        a.slot_q[j] = slot_rz0 + j;
        a.slot_q[k + j] = slot_rr0 + j;
    }
    return launch_block<OP_RESID>(c, k, a);
}

extern "C" int bis_block_cg_update(bis_context *c, int precond, int64_t n, int k, double *R_new, const double *R_old,
                                   const double *AP, double *Z_new, const double *A_D, int slot_rz0, int slot_pAp0,
                                   int slot_rr0, int slot_rz_new0, const double *state) {
    REQ_BLOCK(c, k);
    BIS_REQUIRE(precond == BIS_PRECOND_NONE || precond == BIS_PRECOND_JACOBI,
                "bis_block_cg_update: preconditioner %d not supported (none or jacobi)", precond);
    REQ_BLOCK_VEC(R_new, "R_new"); REQ_BLOCK_VEC(R_old, "R_old"); REQ_BLOCK_VEC(AP, "AP"); REQ_BLOCK_VEC(Z_new, "Z_new");
    BIS_REQUIRE(precond != BIS_PRECOND_JACOBI || A_D, "bis_block_cg_update: jacobi needs A_D");
    REQ_SLOTS(slot_rz0, k, "rz"); REQ_SLOTS(slot_pAp0, k, "pAp"); REQ_SLOTS(slot_rr0, k, "rr");
    REQ_SLOTS(slot_rz_new0, k, "rz_new");
    BlockArgs a = block_args(c, n);
    a.jacobi = precond == BIS_PRECOND_JACOBI;
    a.in0 = R_old; a.in1 = AP; a.D = A_D; a.out0 = R_new; a.out1 = Z_new; a.state = state;
    a.slot_a = slot_rz0; a.slot_b = slot_pAp0;
    for (int j = 0; j < k; ++j) {
        a.slot_q[j] = slot_rr0 + j;
        a.slot_q[k + j] = slot_rz_new0 + j;
    }
    return launch_block<OP_UPDATE>(c, k, a);
}

extern "C" int bis_block_cg_direction_x(bis_context *c, int64_t n, int k, double *P_new, const double *Z_new,
                                        const double *P_old, double *X_new, const double *X_old, int slot_rz_new0,
                                        int slot_rz0, int slot_pAp0, const double *state) {
    REQ_BLOCK(c, k);
    REQ_BLOCK_VEC(P_new, "P_new"); REQ_BLOCK_VEC(Z_new, "Z_new"); REQ_BLOCK_VEC(P_old, "P_old");
    REQ_BLOCK_VEC(X_new, "X_new"); REQ_BLOCK_VEC(X_old, "X_old");
    REQ_SLOTS(slot_rz_new0, k, "rz_new"); REQ_SLOTS(slot_rz0, k, "rz"); REQ_SLOTS(slot_pAp0, k, "pAp");
    BlockArgs a = block_args(c, n);
    a.in0 = Z_new; a.in1 = P_old; a.in2 = X_old; a.out0 = P_new; a.out1 = X_new; a.state = state;
    a.slot_a = slot_rz_new0; a.slot_b = slot_rz0; a.slot_c = slot_pAp0;
    return launch_block<OP_DIRX>(c, k, a);
}

extern "C" int bis_block_cg_status(bis_context *c, int k, int slot_rr0, int max_iters, double *state) {
    REQ_BLOCK(c, k);
    REQ_SLOTS(slot_rr0, k, "rr");
    BIS_REQUIRE(state, "bis_block_cg_status: null state");
    BIS_REQUIRE(max_iters >= 1, "bis_block_cg_status: max_iters = %d < 1", max_iters);
    block_cg_status_kernel<<<1, 32, 0, c->stream>>>(k, c->d_scalars, slot_rr0, max_iters, state);
    BIS_LAUNCH_CHECK(c);
    return 0;
}
