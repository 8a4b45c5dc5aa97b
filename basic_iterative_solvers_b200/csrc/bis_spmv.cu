// bis_spmv.cu -- CRS sparse matrix-vector product (native_spmv,
// kernels.hpp:22-42) and its fused forms:
//   y = A x                                   bis_spmv            kernels.hpp:44-52
//   y = A x ; (y,w) ; (y,y)                   bis_spmv_dot        cg.hpp:16-23, bicgstab.hpp:30-34,48-51
//   tmp = A x ; r = b - tmp ; (r,r)           bis_spmv_residual   kernels.hpp:155-162 + 194-203
//   x_new = (b - (A x_old - D x_old)) / D     bis_spmv_jacobi     jacobi.hpp:27-52
//   out = b - T x                             bis_spmv_sub        gauss_seidel.hpp:30-34
//
// Roofline: HBM.  Algorithmic bytes per launch (SURVEY.md 8(d)):
//   12*nnz + sizeof(row_ptr)*(n+1) + 8*n (x once) + 8*n (y)   [+ 8*n per extra
//   vector an epilogue reads or writes].
//
// Variant 1 ("vector CRS"): LPR lanes cooperate on one row (LPR = 2..32 chosen
// from the mean row length), lanes read consecutive nonzeros (coalesced 8-byte
// val / 4-byte col loads marked evict-first so that x stays cached), x is
// gathered through the read-only path, partial sums are combined by a
// fixed-shape shuffle tree (deterministic), and the epilogue runs on the
// group's first lane.  The grid is persistent (SM count x resident blocks) with
// a static row assignment so the fused dot products are bit-reproducible.
//
// Variant 2 (TMA-staged, thread-per-row) lives in bis_spmv_tma.cu.
#include "bis_device.cuh"
#include "bis_spmv_tma.cuh"
#include "bis_spmv_win.cuh"
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace {

constexpr int SPMV_THREADS = 256;

// variants 1 and 2: one record per rank (deterministic for a given launch shape and rank count; the
// partition-invariant sum is the windowed variant's and the streaming kernels', bis_internal.cuh)
inline void red_set_plain(RedArgs &ra, int total) {
    ra.total_blocks = total;
    ra.n_slab = 1;
    ra.slab_off[0] = 0;
    for (int i = 1; i <= BIS_NSLAB; ++i) ra.slab_off[i] = total;
}

struct SpmvIn {
    const void *rp;
    const int *col;
    const double *val;
    const double *x;       // owned part, indexed by local column
    const double *ghost;   // halo part, indexed by column - n_owned
    int64_t n_owned;
    // rows handled by this launch: [lo1, lo1+cnt1) then [lo2, lo2+cnt2)
    int64_t lo1, cnt1, lo2, cnt2;
};

// Epilogues.  load(r) fetches the per-row operands (issued BEFORE the row's sum is available so
// that their latency overlaps the tile wait / row walk); operator() consumes them.  vectors(x): how
// many n-vectors the epilogue reads or writes besides x (the byte model of spmv_stream_mb).
struct EpiStore {
    static constexpr int NRED = 0;
    double *y;
    int vectors(const double *) const { return 1; }
    __device__ __forceinline__ EpiPre load(int64_t) const { return EpiPre{0.0, 0.0, 0.0}; }
    __device__ __forceinline__ void operator()(int64_t r, double s, const EpiPre &, double *) const { y[r] = s; }
};
struct EpiDot {
    static constexpr int NRED = 2;
    double *y;
    const double *w;
    int vectors(const double *x) const { return 1 + (w != x ? 1 : 0); }
    __device__ __forceinline__ EpiPre load(int64_t r) const { return EpiPre{w[r], 0.0, 0.0}; }
    __device__ __forceinline__ void operator()(int64_t r, double s, const EpiPre &p, double *acc) const {
        y[r] = s;
        acc[0] = fma(s, p.a, acc[0]);
        acc[1] = fma(s, s, acc[1]);
    }
};
struct EpiResid {
    static constexpr int NRED = 1;
    const double *b;
    double *res;
    double *tmp;
    int vectors(const double *) const { return 2 + (tmp ? 1 : 0); }
    __device__ __forceinline__ EpiPre load(int64_t r) const { return EpiPre{b[r], 0.0, 0.0}; }
    __device__ __forceinline__ void operator()(int64_t r, double s, const EpiPre &p, double *acc) const {
        if (tmp) tmp[r] = s;
        double v = sub_rn(p.a, s);   // subtract_vectors with scale 1.0
        res[r] = v;
        acc[0] = fma(v, v, acc[0]);
    }
};
struct EpiJacobi {
    static constexpr int NRED = 0;
    const double *D, *b, *x_old;
    double *x_new;
    int vectors(const double *) const { return 3; }
    __device__ __forceinline__ EpiPre load(int64_t r) const { return EpiPre{D[r], x_old[r], b[r]}; }
    __device__ __forceinline__ void operator()(int64_t r, double s, const EpiPre &p, double *) const {
        double scaled = mul_rn(p.a, p.b);
        double adj = sub_rn(s, scaled);
        x_new[r] = div_rn(sub_rn(p.c, adj), p.a);
    }
};
// Jacobi sweep AND the residual norm of the iterate it starts from, from ONE product A x_old (the reference's loop
// computes A x twice per iteration: jacobi.hpp:27-52 for the sweep, :102-107 for the residual of the same vector one
// harness pass earlier).  Both results are the bits of EpiJacobi / EpiResid.
struct EpiJacobiResid {
    static constexpr int NRED = 1;
    const double *D, *b, *x_old;
    double *x_new;
    double *res;       // may be null
    int vectors(const double *) const { return 3 + (res ? 1 : 0); }
    __device__ __forceinline__ EpiPre load(int64_t r) const { return EpiPre{D[r], x_old[r], b[r]}; }
    __device__ __forceinline__ void operator()(int64_t r, double s, const EpiPre &p, double *acc) const {
        const double scaled = mul_rn(p.a, p.b);
        const double adj = sub_rn(s, scaled);
        x_new[r] = div_rn(sub_rn(p.c, adj), p.a);
        const double v = sub_rn(p.c, s);
        if (res) res[r] = v;
        acc[0] = fma(v, v, acc[0]);
    }
};
struct EpiSub {
    static constexpr int NRED = 0;
    const double *b;
    double *out;
    int vectors(const double *) const { return 2; }
    __device__ __forceinline__ EpiPre load(int64_t r) const { return EpiPre{b[r], 0.0, 0.0}; }
    __device__ __forceinline__ void operator()(int64_t r, double s, const EpiPre &p, double *) const {
        out[r] = sub_rn(p.a, s);
    }
};

// One inner iteration of the two-stage Gauss-Seidel preconditioner (kernels.hpp:321-331):
// tmp = T work ; tmp = (D_inv * -1) * tmp ; output = output + tmp (sum_vectors: one rounding)
struct EpiTwoStage {
    static constexpr int NRED = 0;
    const double *D_inv;
    double *w_out;
    double *out;
    int vectors(const double *) const { return 4; }     // out is read and written
    __device__ __forceinline__ EpiPre load(int64_t r) const { return EpiPre{D_inv[r], out[r], 0.0}; }
    __device__ __forceinline__ void operator()(int64_t r, double s, const EpiPre &p, double *) const {
        const double t = mul_rn(mul_rn(p.a, -1.0), s);
        w_out[r] = t;
        out[r] = fma(1.0, t, p.b);
    }
};

template <typename RP, int LPR, bool GHOST, class Epi>
__global__ void __launch_bounds__(SPMV_THREADS)
spmv_vec_kernel(SpmvIn in, Epi epi, RedArgs ra) {
    constexpr int RPW = 32 / LPR;   // rows per warp per trip
    const RP *__restrict__ rp = static_cast<const RP *>(in.rp);
    const int *__restrict__ col = in.col;
    const double *__restrict__ val = in.val;
    const double *__restrict__ x = in.x;
    const int lane = threadIdx.x & 31;
    const int sub = lane % LPR;
    const int grp = lane / LPR;
    const int64_t warp_global = (int64_t)blockIdx.x * (SPMV_THREADS / 32) + (threadIdx.x >> 5);
    const int64_t total_warps = (int64_t)gridDim.x * (SPMV_THREADS / 32);
    const int64_t total_rows = in.cnt1 + in.cnt2;

    double acc[Epi::NRED > 0 ? Epi::NRED : 1];
#pragma unroll
    for (int q = 0; q < (Epi::NRED > 0 ? Epi::NRED : 1); ++q) acc[q] = 0.0;

    for (int64_t v0 = warp_global * RPW; v0 < total_rows; v0 += total_warps * RPW) {
        const int64_t v = v0 + grp;
        const bool live = v < total_rows;
        const int64_t r = live ? (v < in.cnt1 ? in.lo1 + v : in.lo2 + (v - in.cnt1)) : 0;
        double sum = 0.0;
        if (live) {
            const RP s = rp[r], e = rp[r + 1];
#pragma unroll 4
            for (RP k = s + sub; k < e; k += LPR) {
                const int c = ld_stream(col + k);
                const double a = ld_stream(val + k);
                double xv;
                if (GHOST && c >= in.n_owned) xv = __ldg(in.ghost + (c - in.n_owned));
                else xv = __ldg(x + c);
                sum = fma(a, xv, sum);
            }
        }
#pragma unroll
        for (int o = LPR / 2; o > 0; o >>= 1) sum += __shfl_down_sync(0xffffffffu, sum, o, LPR);
        if (live && sub == 0) epi(r, sum, epi.load(r), acc);
    }
    if constexpr (Epi::NRED > 0) block_reduce_finish<Epi::NRED>(acc, ra);
}

template <typename RP, int LPR, bool GHOST, class Epi>
int launch_one(bis_context *c, const SpmvIn &in, const Epi &epi, RedArgs &ra, int *blocks_out) {
    static int occ = 0;
    if (!occ) {
        BIS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(
            &occ, spmv_vec_kernel<RP, LPR, GHOST, Epi>, SPMV_THREADS, 0));
        if (occ < 1) occ = 1;
    }
    const int64_t rows = in.cnt1 + in.cnt2;
    constexpr int rows_per_block = (SPMV_THREADS / 32) * (32 / LPR);
    int cap = c->sm_count * occ;
    if (cap > BIS_MAX_RED_BLOCKS / 4) cap = BIS_MAX_RED_BLOCKS / 4;
    int blocks = bis_blocks_for(rows, rows_per_block, cap);
    *blocks_out = blocks;
    if (Epi::NRED > 0 && ra.finalize) red_set_plain(ra, ra.block_offset + blocks);
    spmv_vec_kernel<RP, LPR, GHOST, Epi><<<blocks, SPMV_THREADS, 0, c->stream>>>(in, epi, ra);
    BIS_LAUNCH_CHECK(c);
    return 0;
}

template <typename RP, bool GHOST, class Epi>
int launch_lanes(bis_context *c, int lanes, const SpmvIn &in, const Epi &epi, RedArgs &ra, int *nb) {
    switch (lanes) {
    case 2: return launch_one<RP, 2, GHOST, Epi>(c, in, epi, ra, nb);
    case 4: return launch_one<RP, 4, GHOST, Epi>(c, in, epi, ra, nb);
    case 8: return launch_one<RP, 8, GHOST, Epi>(c, in, epi, ra, nb);
    case 16: return launch_one<RP, 16, GHOST, Epi>(c, in, epi, ra, nb);
    default: return launch_one<RP, 32, GHOST, Epi>(c, in, epi, ra, nb);
    }
}

int pick_lanes(const bis_context *c, const bis_matrix *A) {
    if (c->opt_spmv_lanes >= 2) {
        int l = 2;
        while (l < c->opt_spmv_lanes && l < 32) l <<= 1;
        return l;
    }
    // ~4 nonzeros per lane: 27/row -> 8 lanes, 7/row -> 2, 13/row -> 4
    double m = A->mean_row;
    int l = 2;
    while (l < 32 && l * 4 < m) l <<= 1;
    return l;
}

template <bool GHOST, class Epi>
int launch_rp(bis_context *c, const bis_matrix *A, const SpmvIn &in, const Epi &epi, RedArgs &ra,
              int *nb) {
    const int lanes = pick_lanes(c, A);
    if (A->rp_bytes == 8) return launch_lanes<int64_t, GHOST, Epi>(c, lanes, in, epi, ra, nb);
    return launch_lanes<int32_t, GHOST, Epi>(c, lanes, in, epi, ra, nb);
}

} // namespace

// ---- variant 2 (TMA-staged, thread per row): plan + launch ------------------------------
namespace {

bool tma_plan(const bis_context *c, const bis_matrix *A, tma::Plan *p) {
    if (c->opt_spmv_variant == 1) return false;
    if (A->max_row < 1 || A->max_row > 96) return false;
    // Measured on HPCG-512 (tools/tune_spmv.py, profiles/): small tiles with two stages and
    // several resident CTAs per SM beat one big CTA -- the tile is consumed in latency-bound
    // phases, and co-resident CTAs overlap them.  Default: ~20 KB per stage.
    const size_t budget = (size_t)(c->opt_spmv_smem_kb > 0 ? c->opt_spmv_smem_kb : 44) << 10;
    const int max_stages = c->opt_spmv_stages > 0 ? c->opt_spmv_stages : 2;
    for (int R : {256, 128, 64, 32}) {
        if (c->opt_spmv_rows > 0 && R != c->opt_spmv_rows) continue;
        const int cap = (R * A->max_row + 8 + 3) & ~3;
        const size_t stage = (size_t)cap * 12;
        int nstage = (int)((budget - 128) / stage);
        if (nstage > max_stages) nstage = max_stages;
        if (nstage > tma::MAX_STAGES) nstage = tma::MAX_STAGES;
        if (nstage < 2) continue;
        int mult = c->opt_spmv_mult > 0 ? c->opt_spmv_mult : 2;
        while (R * mult > 1024) mult >>= 1;
        p->threads = R * mult;
        p->rows = R;
        p->cap = cap;
        p->nstage = nstage;
        p->smem_bytes = 128 + stage * nstage;
        return true;
    }
    return false;
}

template <typename RP, bool GHOST, class Epi>
int launch_tma(bis_context *c, const tma::Plan &p, SpmvTmaIn in, const Epi &epi, RedArgs &ra, int *nb) {
    auto kern = spmv_tma_kernel<RP, GHOST, Epi>;
    BIS_CHECK(bis_ensure_dynamic_smem(c, reinterpret_cast<const void *>(kern), p.smem_bytes));
    int occ = 1;
    BIS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, p.threads, p.smem_bytes));
    if (occ < 1) occ = 1;
    const int64_t n_tiles = (in.cnt + p.rows - 1) / p.rows;
    int64_t grid = (int64_t)c->sm_count * occ;
    if (grid > n_tiles) grid = n_tiles;
    if (grid < 1) grid = 1;
    in.tiles_per_cta = (n_tiles + grid - 1) / grid;
    if (in.tiles_per_cta < 1) in.tiles_per_cta = 1;
    in.cap = p.cap;
    in.nstage = p.nstage;
    in.interleave = c->opt_spmv_blocked ? 0 : 1;
    in.rows = p.rows;
    *nb = (int)grid;
    if (Epi::NRED > 0 && ra.finalize) red_set_plain(ra, ra.block_offset + (int)grid);
    kern<<<(unsigned)grid, p.threads, p.smem_bytes, c->stream>>>(in, epi, ra);
    BIS_LAUNCH_CHECK(c);
    return 0;
}

struct Segment {
    int64_t lo, cnt;
    bool ghost;
};

// One contiguous row range with either variant.
template <class Epi>
int launch_segment(bis_context *c, const bis_matrix *A, const double *x, const Segment &sg, const Epi &epi,
                   RedArgs &ra, int *nb) {
    tma::Plan plan;
    if (tma_plan(c, A, &plan)) {
        SpmvTmaIn in;
        in.rp = A->d_rp; in.col = A->d_col; in.val = A->d_val; in.x = x;
        in.ghost = A->halo.cur_ghost; in.n_owned = A->n_cols;
        in.lo = sg.lo; in.cnt = sg.cnt;
        in.tiles_per_cta = 1; in.cap = 0; in.nstage = 0; in.interleave = 1; in.rows = 0;
        if (A->rp_bytes == 8)
            return sg.ghost ? launch_tma<int64_t, true, Epi>(c, plan, in, epi, ra, nb)
                            : launch_tma<int64_t, false, Epi>(c, plan, in, epi, ra, nb);
        return sg.ghost ? launch_tma<int32_t, true, Epi>(c, plan, in, epi, ra, nb)
                        : launch_tma<int32_t, false, Epi>(c, plan, in, epi, ra, nb);
    }
    SpmvIn in;
    in.rp = A->d_rp; in.col = A->d_col; in.val = A->d_val; in.x = x;
    in.ghost = A->halo.cur_ghost; in.n_owned = A->n_cols;
    in.lo1 = sg.lo; in.cnt1 = sg.cnt; in.lo2 = 0; in.cnt2 = 0;
    return sg.ghost ? launch_rp<true, Epi>(c, A, in, epi, ra, nb) : launch_rp<false, Epi>(c, A, in, epi, ra, nb);
}

} // namespace

// ---- variant 3 (windowed x, everything by TMA): lazy format build, plan, launch ----------------
namespace {

int win_free(bis_matrix *A) {
    WinFormat &w = A->win;
    cudaFree(w.d_seg_start); cudaFree(w.d_seg_len); cudaFree(w.d_seg_off); cudaFree(w.d_nseg); cudaFree(w.d_lidx);
    cudaFree(w.d_order); cudaFree(w.d_vidx); cudaFree(w.d_vdict);
    w.d_seg_start = nullptr; w.d_seg_len = nullptr; w.d_seg_off = nullptr; w.d_nseg = nullptr; w.d_lidx = nullptr;
    w.d_order = nullptr; w.d_vidx = nullptr; w.d_vdict = nullptr;
    w.dict_state = 0; w.n_dict = 0;
    return 0;
}

// ---- value dictionary (WinFormat::d_vidx / d_vdict) ------------------------------------------------
// Pass 1 collects the distinct bit patterns of val[] (a block keeps the ones it has met in shared memory, so the global
// table sees each pattern once per block, not once per nonzero) and gives up beyond 256; the host sorts them; pass 2
// writes the index of every value.  A matrix with many distinct values leaves pass 1 after a few thousand nonzeros.
constexpr int VD_SLOTS = 1024;                         // global table (power of two, > 2 * 256)
constexpr int VD_LOCAL = 512;                          // per-block table
constexpr unsigned long long VD_EMPTY = ~0ull;         // a NaN pattern: a matrix that holds it gets no dictionary

__device__ __forceinline__ unsigned int vd_hash(unsigned long long v) {
    v ^= v >> 33;
    v *= 0xff51afd7ed558ccdull;
    v ^= v >> 29;
    return (unsigned int)v;
}

__global__ void __launch_bounds__(256) vdict_collect_kernel(int64_t nnz, const double *val, unsigned long long *slots, int *state) {
    __shared__ unsigned long long s_slots[VD_LOCAL];
    __shared__ int s_count;
    for (int i = threadIdx.x; i < VD_LOCAL; i += blockDim.x) s_slots[i] = VD_EMPTY;
    if (threadIdx.x == 0) s_count = 0;
    __syncthreads();
    int it = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x, ++it) {
        if (*reinterpret_cast<volatile int *>(&s_count) > 256) return;
        if ((it & 63) == 0 && *reinterpret_cast<volatile int *>(state + 1)) return;    // somebody gave up (looked at rarely: one address)
        const unsigned long long v = (unsigned long long)__double_as_longlong(val[i]);
        if (v == VD_EMPTY) {
            atomicExch(state + 1, 1);
            return;
        }
        unsigned int h = vd_hash(v) & (VD_LOCAL - 1);
        bool fresh = false;
        for (int probe = 0; probe < VD_LOCAL; ++probe) {
            const unsigned long long cur = *reinterpret_cast<volatile unsigned long long *>(&s_slots[h]);
            if (cur == v) break;
            if (cur == VD_EMPTY) {
                const unsigned long long old = atomicCAS(&s_slots[h], VD_EMPTY, v);
                if (old == VD_EMPTY) {
                    fresh = true;
                    atomicAdd(&s_count, 1);
                    break;
                }
                if (old == v) break;
            }
            h = (h + 1) & (VD_LOCAL - 1);
        }
        if (!fresh) continue;
        // new to this block: into the global table
        unsigned int g = vd_hash(v) & (VD_SLOTS - 1);
        for (int probe = 0; probe < VD_SLOTS; ++probe) {
            const unsigned long long cur = *reinterpret_cast<volatile unsigned long long *>(&slots[g]);
            if (cur == v) break;
            if (cur == VD_EMPTY) {
                const unsigned long long old = atomicCAS(&slots[g], VD_EMPTY, v);
                if (old == VD_EMPTY) {
                    if (atomicAdd(state, 1) + 1 > 256) atomicExch(state + 1, 1);
                    break;
                }
                if (old == v) break;
            }
            g = (g + 1) & (VD_SLOTS - 1);
        }
    }
}

__global__ void __launch_bounds__(256) vdict_index_kernel(int64_t nnz, const double *val, const double *dict, int n_dict,
                                                          unsigned char *vidx, int *missing) {
    __shared__ unsigned long long s_d[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x)
        s_d[i] = i < n_dict ? (unsigned long long)__double_as_longlong(dict[i]) : VD_EMPTY;
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned long long v = (unsigned long long)__double_as_longlong(val[i]);
        int lo = 0, hi = n_dict - 1;
        while (lo < hi) {           // first entry >= v (ascending bit patterns)
            const int mid = (lo + hi) >> 1;
            if (s_d[mid] < v) lo = mid + 1;
            else hi = mid;
        }
        if (s_d[lo] != v) atomicExch(missing, 1);
        vidx[i] = (unsigned char)lo;
    }
}

// Builds the dictionary of A's values when there are at most 256 distinct ones (dict_state 1), else dict_state -1.
int win_build_dict(bis_context *c, const bis_matrix *A) {
    WinFormat &w = A->win;
    if (w.dict_state != 0 || !c->opt_spmv_vdict) return 0;     // (switched on later, it is built then)
    w.dict_state = -1;
    if (A->nnz == 0 || !A->d_val) return 0;
    unsigned long long *d_slots = nullptr;
    int *d_state = nullptr;
    BIS_CUDA(bis_cuda_malloc(&d_slots, sizeof(unsigned long long) * VD_SLOTS));
    BIS_CUDA(bis_cuda_malloc(&d_state, 3 * sizeof(int)));
    BIS_CUDA(cudaMemsetAsync(d_slots, 0xFF, sizeof(unsigned long long) * VD_SLOTS, c->stream));
    BIS_CUDA(cudaMemsetAsync(d_state, 0, 3 * sizeof(int), c->stream));
    const int blocks = bis_blocks_for(A->nnz, 256 * 16, c->sm_count * 8);
    vdict_collect_kernel<<<blocks, 256, 0, c->stream>>>(A->nnz, A->d_val, d_slots, d_state);
    BIS_LAUNCH_CHECK(c);
    std::vector<unsigned long long> slots(VD_SLOTS);
    int state[3] = {0, 0, 0};
    BIS_CUDA(cudaMemcpyAsync(slots.data(), d_slots, sizeof(unsigned long long) * VD_SLOTS, cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaMemcpyAsync(state, d_state, sizeof state, cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(d_slots);
    std::vector<unsigned long long> pats;
    for (unsigned long long v : slots)
        if (v != VD_EMPTY) pats.push_back(v);
    if (state[1] != 0 || pats.empty() || pats.size() > 256) {
        cudaFree(d_state);
        return 0;
    }
    std::sort(pats.begin(), pats.end());
    double dict[256] = {};
    for (size_t i = 0; i < pats.size(); ++i) memcpy(&dict[i], &pats[i], sizeof(double));
    // the index array is an acceleration structure: it is built only while an eighth of the device memory stays free
    // after it, so that what the solver allocates later (vectors, triangular factors) is not crowded out by it
    size_t fr = 0, tot = 0;
    if (cudaMemGetInfo(&fr, &tot) != cudaSuccess || (size_t)A->nnz + 32 + tot / 8 > fr) {
        cudaGetLastError();
        cudaFree(d_state);
        return 0;
    }
    if (cudaMalloc(&w.d_vidx, (size_t)A->nnz + 32) != cudaSuccess) {     // no room for the index array: the values are streamed
        cudaGetLastError();
        w.d_vidx = nullptr;
        cudaFree(d_state);
        return 0;
    }
    BIS_CUDA(bis_cuda_malloc(&w.d_vdict, sizeof(double) * 256));
    BIS_CUDA(cudaMemcpyAsync(w.d_vdict, dict, sizeof dict, cudaMemcpyHostToDevice, c->stream));
    BIS_CUDA(cudaMemsetAsync(w.d_vidx + A->nnz, 0, 32, c->stream));
    vdict_index_kernel<<<blocks, 256, 0, c->stream>>>(A->nnz, A->d_val, w.d_vdict, (int)pats.size(), w.d_vidx, d_state + 2);
    BIS_LAUNCH_CHECK(c);
    BIS_CUDA(cudaMemcpyAsync(state, d_state, sizeof state, cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(d_state);
    if (state[2] != 0) {        // cannot happen unless val[] changed between the two passes
        cudaFree(w.d_vidx); cudaFree(w.d_vdict);
        w.d_vidx = nullptr; w.d_vdict = nullptr;
        return 0;
    }
    w.n_dict = (int)pats.size();
    w.dict_state = 1;
    return 0;
}

// ---- tile order (bis_spmv_win.cuh: WinOrderArgs) ---------------------------------------------------
// flags of a tile relative to ITS virtual slab [lo, hi) (local rows): bit 0 some column below the slab,
// bit 1 some column at or above its end, bit 2 some ghost column.  Ghost columns are ordered by global id:
// the first n_low_ghost of them belong to lower ranks.  One warp per tile.
template <typename RP>
__global__ void __launch_bounds__(256) tile_flags_kernel(int64_t n_tiles, int R, int64_t n_rows, const RP *rp, const int *col,
                                                         int n_owned, int n_low_ghost, int n_slab, const int64_t *slab_row,
                                                         unsigned char *flags) {
    const int lane = threadIdx.x & 31;
    for (int64_t t = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); t < n_tiles; t += (int64_t)gridDim.x * 8) {
        const int64_t r0 = t * R;
        int64_t r1 = r0 + R;
        if (r1 > n_rows) r1 = n_rows;
        int i = 0;
        while (i + 1 < n_slab && r0 >= slab_row[i + 1]) ++i;
        const int64_t lo = slab_row[i], hi = slab_row[i + 1];
        unsigned int f = 0;
        for (int64_t k = (int64_t)rp[r0] + lane; k < (int64_t)rp[r1]; k += 32) {
            const int cc = col[k];
            if (cc >= n_owned) f |= 4u | ((cc - n_owned) < n_low_ghost ? 1u : 2u);
            else if (cc < lo) f |= 1u;
            else if (cc >= hi) f |= 2u;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) f |= __shfl_xor_sync(0xffffffffu, f, o);
        if (lane == 0) flags[t] = (unsigned char)f;
    }
}

// Builds the processing order of the tiles (see bis_spmv_win.cuh).  Host work is O(n_tiles).
int win_build_order(bis_context *c, const bis_matrix *A) {
    WinFormat &w = A->win;
    const int64_t nt = w.n_tiles;
    const int R = w.R;
    // virtual slabs: the context's partition when it describes this matrix and its slabs start on tiles
    RowPartition part = bis_partition_for(c, A->n_rows);
    bool inv = part.invariant && part.n_global == A->n_rows_global && part.row_begin == A->row_begin && A->triangular == 0;
    for (int i = 0; inv && i < part.n_slab; ++i)
        if (part.slab_row[i] % R != 0) inv = false;
    if (!inv) {
        part.n_slab = 1;
        part.slab_first = 0;
        part.slab_row[0] = 0;
        part.slab_row[1] = A->n_rows;
    }
    int64_t *d_slab = nullptr;
    unsigned char *d_flags = nullptr;
    BIS_CUDA(bis_cuda_malloc(&d_slab, sizeof(int64_t) * (BIS_NSLAB + 1)));
    BIS_CUDA(bis_cuda_malloc(&d_flags, (size_t)nt));
    BIS_CUDA(cudaMemcpyAsync(d_slab, part.slab_row, sizeof(int64_t) * (part.n_slab + 1), cudaMemcpyHostToDevice, c->stream));
    const int n_low = A->distributed ? (int)A->halo.recv_off[c->rank] : 0;
    const int blocks = bis_blocks_for(nt, 8, c->sm_count * 16);
    if (A->rp_bytes == 8)
        tile_flags_kernel<int64_t><<<blocks, 256, 0, c->stream>>>(nt, R, A->n_rows, static_cast<const int64_t *>(A->d_rp), A->d_col,
                                                                  (int)A->n_cols, n_low, part.n_slab, d_slab, d_flags);
    else
        tile_flags_kernel<int32_t><<<blocks, 256, 0, c->stream>>>(nt, R, A->n_rows, static_cast<const int32_t *>(A->d_rp), A->d_col,
                                                                  (int)A->n_cols, n_low, part.n_slab, d_slab, d_flags);
    BIS_LAUNCH_CHECK(c);
    std::vector<unsigned char> flags((size_t)nt);
    BIS_CUDA(cudaMemcpyAsync(flags.data(), d_flags, (size_t)nt, cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(d_flags);
    cudaFree(d_slab);
    // y-blocked traversal of the interiors: between two uses of a plane of x (by the tiles of plane z-1, z
    // and z+1) the grid streams two planes of matrix data; when that no longer fits the L2 the planes are
    // cut into nb blocks of tiles and the slab is swept block by block through z (SpMV "x planes in L2").
    int nb = 1;
    int64_t Pt = 0, Bt = 0;
    const int64_t plane = A->grid_nx * A->grid_ny;
    if (plane > 0 && plane % R == 0 && A->row_begin % plane == 0) {
        Pt = plane / R;
        const double bytes_per_row = 10.0 * A->mean_row + 32.0;
        const double budget = 1.0e6 * (c->opt_spmv_l2_mb > 0 ? c->opt_spmv_l2_mb : 40);   // bytes streamed between two uses of an x value
        const double two_planes = 2.0 * (double)plane * bytes_per_row;
        if (two_planes > budget) nb = (int)((two_planes + budget - 1) / budget);
        if (nb > Pt) nb = (int)Pt;
        Bt = (Pt + nb - 1) / nb;
    }
    w.traversal_blocks = nb;
    std::vector<int> order;
    order.reserve((size_t)nt);
    std::vector<int> interior, lowv, highv;
    const int64_t tile0 = A->row_begin / R;   // global index of local tile 0 (row_begin % R == 0 when invariant)
    w.pos0[0] = 0;
    for (int i = 0; i < part.n_slab; ++i) {
        const int64_t t0 = part.slab_row[i] / R, t1 = (part.slab_row[i + 1] + R - 1) / R;
        interior.clear(); lowv.clear(); highv.clear();
        for (int64_t t = t0; t < t1; ++t) {
            const unsigned char f = flags[(size_t)t];
            const int e = (int)t | ((f & 4) ? WIN_ORDER_GHOST : 0);
            if (f & 2) highv.push_back(e);
            else if (f & 1) lowv.push_back(e);
            else interior.push_back(e);
        }
        if (nb > 1) {
            // key (block, plane), ascending tile inside: a stable counting pass per block keeps it O(n)
            std::vector<int> tmp;
            tmp.reserve(interior.size());
            for (int b = 0; b < nb; ++b)
                for (int e : interior) {
                    const int64_t tg = tile0 + (e & ~WIN_ORDER_GHOST);
                    if ((tg % Pt) / Bt == b) tmp.push_back(e);
                }
            interior.swap(tmp);
        }
        order.insert(order.end(), interior.begin(), interior.end());
        order.insert(order.end(), lowv.begin(), lowv.end());
        order.insert(order.end(), highv.begin(), highv.end());
        w.pos0[i + 1] = (int)order.size();
    }
    for (int i = part.n_slab + 1; i <= BIS_NSLAB; ++i) w.pos0[i] = w.pos0[part.n_slab];
    w.n_slab = part.n_slab;
    w.slab_first = part.slab_first;
    w.invariant = inv;
    BIS_CUDA(bis_cuda_malloc(&w.d_order, sizeof(int) * (size_t)(nt > 0 ? nt : 1)));
    BIS_CUDA(cudaMemcpyAsync(w.d_order, order.data(), sizeof(int) * (size_t)nt, cudaMemcpyHostToDevice, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

// Builds A->win on first use.  Returns 0 and sets win.state = 1 (usable) or -1 (some tile needs more
// than WIN_MAXSEG windows: unstructured matrix, variant 2 is used instead).
int win_build(bis_context *c, const bis_matrix *A) {
    WinFormat &w = A->win;
    if (w.state != 0) return 0;
    w.state = -1;
    if (A->n_rows == 0 || A->nnz == 0 || A->max_row < 1) return 0;
    int R = c->opt_win_rows;
    if (R != 32 && R != 64 && R != 128 && R != 256) {
        R = 128;
        while (R > 32 && (size_t)R * A->max_row * 10 > (size_t)40 << 10) R >>= 1;   // ~<= 40 KB of val+lidx per stage
    }
    if ((size_t)R * A->max_row * 10 > (size_t)96 << 10) return 0;                     // rows too long for a tile
    int sort_cap = 1;
    while (sort_cap < R * A->max_row) sort_cap <<= 1;
    const int64_t n_tiles = (A->n_rows + R - 1) / R;
    int *d_status = nullptr;
    BIS_CUDA(bis_cuda_malloc(&d_status, 2 * sizeof(int)));
    BIS_CUDA(cudaMemsetAsync(d_status, 0, 2 * sizeof(int), c->stream));
    BIS_CUDA(bis_cuda_malloc(&w.d_seg_start, sizeof(int) * (size_t)n_tiles * WIN_MAXSEG));
    BIS_CUDA(bis_cuda_malloc(&w.d_seg_len, sizeof(unsigned short) * (size_t)n_tiles * WIN_MAXSEG));
    BIS_CUDA(bis_cuda_malloc(&w.d_seg_off, sizeof(unsigned short) * (size_t)n_tiles * WIN_MAXSEG));
    BIS_CUDA(bis_cuda_malloc(&w.d_nseg, sizeof(int) * (size_t)n_tiles));
    BIS_CUDA(bis_cuda_malloc(&w.d_lidx, sizeof(unsigned short) * ((size_t)A->nnz + 32)));
    WinBuildArgs a;
    a.rp = A->d_rp; a.col = A->d_col; a.n_rows = A->n_rows; a.n_owned = A->n_cols; a.R = R; a.sort_cap = sort_cap;
    a.seg_start = w.d_seg_start; a.seg_len = w.d_seg_len; a.seg_off = w.d_seg_off; a.nseg = w.d_nseg;
    a.lidx = w.d_lidx; a.status = d_status;
    const size_t smem = sizeof(int) * (size_t)sort_cap;
    if (A->rp_bytes == 8) {
        BIS_CUDA(cudaFuncSetAttribute(win_build_kernel<int64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        win_build_kernel<int64_t><<<(unsigned)n_tiles, WIN_BUILD_THREADS, smem, c->stream>>>(a);
    } else {
        BIS_CUDA(cudaFuncSetAttribute(win_build_kernel<int32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        win_build_kernel<int32_t><<<(unsigned)n_tiles, WIN_BUILD_THREADS, smem, c->stream>>>(a);
    }
    BIS_LAUNCH_CHECK(c);
    int status[2] = {0, 0};
    BIS_CUDA(cudaMemcpyAsync(status, d_status, sizeof status, cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(d_status);
    if (status[1] != 0) {
        win_free(const_cast<bis_matrix *>(A));
        return 0;
    }
    w.R = R;
    w.cap = (R * A->max_row + 32 + 15) & ~15;      // a tile's nonzeros + the alignment padding of its copies (up to 15 either side)
    w.xcap = (status[0] + 1) & ~1;
    if (w.xcap < 2) w.xcap = 2;
    w.n_tiles = n_tiles;
    if (win_build_order(c, A) != 0) {
        win_free(const_cast<bis_matrix *>(A));
        return 1;
    }
    w.state = 1;
    return 0;
}

struct WinPlan {
    int nstage;
    int ngroups;
    int stage_bytes;
    size_t smem_bytes;
};

bool win_plan(const bis_context *c, const bis_matrix *A, WinPlan *p) {
    const WinFormat &w = A->win;
    const bool dict = w.dict_state == 1 && c->opt_spmv_vdict;
    size_t stage = (size_t)w.cap * (dict ? 1 : 8) + (size_t)w.xcap * 8 + (size_t)(w.R + 4) * 8 + (size_t)w.cap * 2;
    stage = (stage + 127) & ~(size_t)127;
    const size_t budget = (size_t)(c->opt_spmv_smem_kb > 0 ? c->opt_spmv_smem_kb : 110) << 10;
    int nstage = (int)((budget - 128) / stage);
    const int max_stages = c->opt_spmv_stages > 0 ? c->opt_spmv_stages : 4;
    if (nstage > max_stages) nstage = max_stages;
    if (nstage > tma::MAX_STAGES) nstage = tma::MAX_STAGES;
    if (nstage < 2) {
        if (128 + 2 * stage > ((size_t)220 << 10)) return false;
        nstage = 2;
    }
    // CTA size: at most 320 threads (two or more CTAs per SM) unless the tile itself is 256 rows long
    const int max_threads = w.R > 128 ? WIN_MAX_THREADS : 320;
    // one consumer group per stage ...
    int ngroups = nstage;
    while (ngroups > 2 && w.R * ngroups + 32 > max_threads) --ngroups;
    if (w.R * ngroups + 32 > max_threads) return false;
    // ... unless the stages are small (value dictionary: a 128-row tile of a 27-point matrix is 21 KB instead of 44): then
    // the two groups of a CTA are fed by a deeper pipeline.  With two stages the kernel was bound by the latency of a
    // tile (two tiles in flight per CTA whatever their size: 5.5 ms at HPCG-512); the groups, and with them the sets of
    // tiles a thread accumulates over, are those of the value-streaming launch, so fused dot products keep their bits.
    if (dict && nstage > ngroups) nstage -= nstage % ngroups;
    else nstage = ngroups;
    p->nstage = nstage;
    p->ngroups = ngroups;
    p->stage_bytes = (int)stage;
    p->smem_bytes = 128 + stage * nstage;
    return true;
}

// One launch over all tiles in table order.  FUSED: the kernel also performs the halo exchange (pack +
// publish before the sweep, the senders' flags checked at the first tile that reads ghosts).
template <typename RP, class Epi, bool FUSED>
int launch_win(bis_context *c, const bis_matrix *A, const WinPlan &p, const double *x, const Epi &epi, RedArgs &ra) {
    auto kern = spmv_win_kernel<RP, Epi, FUSED>;
    BIS_CHECK(bis_ensure_dynamic_smem(c, reinterpret_cast<const void *>(kern), p.smem_bytes));
    const WinFormat &w = A->win;
    const int threads = w.R * p.ngroups + 32;         // the consumer groups + the producer warp
    int occ = 1;
    BIS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, p.smem_bytes));
    if (occ < 1) occ = 1;
    // logical grid G: a property of the device and the tile shape, NOT of the tile count (partition invariance);
    // fewer CTAs are launched when there are fewer tiles -- the missing ones would have had no work
    const int G = c->sm_count * occ;
    int64_t grid = G;
    if (grid > w.n_tiles) grid = w.n_tiles;
    if (grid < 1) grid = 1;
    SpmvWinIn in;
    in.rp = A->d_rp; in.val = A->d_val; in.lidx = w.d_lidx;
    in.seg_start = w.d_seg_start; in.seg_len = w.d_seg_len; in.seg_off = w.d_seg_off; in.nseg = w.d_nseg;
    in.x = x; in.n_rows = A->n_rows;
    in.ord.order = w.d_order;
    in.ord.n_slab = w.n_slab;
    for (int i = 0; i <= BIS_NSLAB; ++i) in.ord.pos0[i] = w.pos0[i];
    in.ord.G = G;
    in.ord.part_stride = (int)grid;
    in.R = w.R; in.cap = w.cap; in.xcap = w.xcap; in.nstage = p.nstage; in.ngroups = p.ngroups; in.stage_bytes = p.stage_bytes;
    const bool dict = w.dict_state == 1 && c->opt_spmv_vdict;
    in.vidx = dict ? w.d_vidx : nullptr;
    in.vdict = dict ? w.d_vdict : nullptr;
    in.n_dict = dict ? w.n_dict : 0;
    in.val_region = dict ? w.cap : w.cap * 8;
    in.amask = dict ? 15 : 7;
    c->last_spmv_value_bytes = dict ? 1 : 8;
    // the launch's compulsory HBM bytes in this format: value (8 B or a 1-byte dictionary index) and 16-bit column id
    // per nonzero, the row_ptr slices, x once, and the vectors of the epilogue (the x windows are re-read from L2)
    c->last_spmv_stream_bytes = (int64_t)(dict ? 3 : 10) * A->nnz + (int64_t)A->rp_bytes * (A->n_rows + 1) +
                                8 * (A->n_cols + (int64_t)epi.vectors(x) * A->n_rows);
#ifdef BIS_PERF_DEBUG
    in.debug = c->opt_spmv_debug;
    in.stamps = nullptr;
    const char *stamp_file = (c->opt_spmv_debug & 4) ? getenv("BIS_SPMV_STAMPS") : nullptr;
    if (stamp_file) {
        BIS_CUDA(bis_cuda_malloc(&in.stamps, sizeof(unsigned long long) * WIN_NSTAMP));
        BIS_CUDA(cudaMemsetAsync(in.stamps, 0, sizeof(unsigned long long) * WIN_NSTAMP, c->stream));
    }
#endif
    ra.finalize = 1;
    ra.block_offset = 0;
    if (Epi::NRED > 0) {
        RowPartition part;
        part.invariant = w.invariant;
        part.n_slab = w.n_slab;
        part.slab_first = w.slab_first;
        int off[BIS_NSLAB + 1];
        for (int i = 0; i <= w.n_slab; ++i) off[i] = i * (int)grid;
        bis_red_set_slabs(c, ra, part, off, w.n_slab * (int)grid);
        if (!w.invariant) {
            // one record per rank, but the partials are still laid out per slab: add them all
            ra.n_slab = 1;
            ra.slab_off[0] = 0;
            for (int i = 1; i <= BIS_NSLAB; ++i) ra.slab_off[i] = w.n_slab * (int)grid;
        }
    }
    if constexpr (FUSED) {
        HaloFuse hf;
        BIS_CHECK(bis_halo_fuse_args(c, A, &hf));
        in.ghost = A->halo.cur_ghost;
        kern<<<(unsigned)grid, threads, p.smem_bytes, c->stream>>>(in, epi, ra, hf);
    } else {
        in.ghost = A->halo.cur_ghost;
        kern<<<(unsigned)grid, threads, p.smem_bytes, c->stream>>>(in, epi, ra, NoHaloFuse{});
    }
    BIS_LAUNCH_CHECK(c);
#ifdef BIS_PERF_DEBUG
    if (in.stamps) {
        unsigned long long h[WIN_NSTAMP];
        BIS_CUDA(cudaMemcpyAsync(h, in.stamps, sizeof h, cudaMemcpyDeviceToHost, c->stream));
        BIS_CUDA(cudaStreamSynchronize(c->stream));
        h[WIN_NSTAMP - 1] = (unsigned long long)grid;
        if (FILE *f = fopen(stamp_file, "ab")) {
            fwrite(h, sizeof(unsigned long long), WIN_NSTAMP, f);
            fclose(f);
        }
        cudaFree(in.stamps);
    }
#endif
    return 0;
}

} // namespace

int bis_spmv_prepare(bis_context *c, const bis_matrix *A) {
    if (c->opt_spmv_variant != 0 && c->opt_spmv_variant != 3) return 0;
    BIS_CHECK(win_build(c, A));
    if (A->win.state == 1) BIS_CHECK(win_build_dict(c, A));
    return 0;
}

void bis_win_values_changed(const bis_matrix *A) {
    WinFormat &w = A->win;
    cudaFree(w.d_vidx);
    cudaFree(w.d_vdict);
    w.d_vidx = nullptr;
    w.d_vdict = nullptr;
    w.n_dict = 0;
    w.dict_state = 0;       // looked at again by the next SpMV
}

// Shared driver: halo exchange (distributed) overlapped with the interior rows.
template <class Epi>
static int spmv_driver(bis_context *c, const bis_matrix *A, const double *x, const Epi &epi,
                       int slot_a, int slot_b) {
    BIS_REQUIRE(c && A && x, "spmv: null argument");
    BIS_REQUIRE_CRS(A);
    BisNvtxRange nvtx_range("spmv");
    BIS_CUDA(cudaSetDevice(c->device));
    RedArgs ra = bis_red_args(c, slot_a, slot_b);
    // variant: 3 (windowed x) when the matrix is representable and x is 16-byte aligned (the reference
    // offsets x, gmres.hpp:168: &V[k*N] with odd N is not), else 2 (TMA tiles + gathers), else 1
    bool use_win = false;
    WinPlan wplan;
    if ((c->opt_spmv_variant == 0 || c->opt_spmv_variant == 3) && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
        BIS_CHECK(win_build(c, A));
        if (A->win.state == 1) BIS_CHECK(win_build_dict(c, A));
        use_win = A->win.state == 1 && win_plan(c, A, &wplan);
    }
    BIS_REQUIRE(use_win || c->opt_spmv_variant != 3,
                "spmv_variant=3 forced, but the matrix has no window representation or x is not 16-byte aligned");
    BIS_CHECK(bis_prof_begin(c, BIS_PROF_SPMV));
    if (use_win) {
        const bool fused = A->distributed && c->opt_spmv_fused && c->peer_on && c->opt_dist_p2p && A->halo.peer_ready;
        if (fused) {
            if (A->rp_bytes == 8) BIS_CHECK((launch_win<int64_t, Epi, true>(c, A, wplan, x, epi, ra)));
            else BIS_CHECK((launch_win<int32_t, Epi, true>(c, A, wplan, x, epi, ra)));
        } else {
            // separate exchange (NCCL transport, or spmv_fused = 0): the sweep starts when the ghosts are in
            if (A->distributed) {
                BIS_CHECK(bis_halo_exchange_begin(c, A, x));
                BIS_CHECK(bis_halo_exchange_end(c, A));
            }
            if (A->rp_bytes == 8) BIS_CHECK((launch_win<int64_t, Epi, false>(c, A, wplan, x, epi, ra)));
            else BIS_CHECK((launch_win<int32_t, Epi, false>(c, A, wplan, x, epi, ra)));
        }
        BIS_CHECK(bis_prof_end(c, BIS_PROF_SPMV));
        if (Epi::NRED > 0) BIS_CHECK(bis_reduce_finish(c, slot_a, slot_b));
        return 0;
    }
    // work list: row ranges (variants 1, 2) or tile ranges (variant 3); `ghost` = needs the halo
    Segment seg[3];
    int nseg = 0;
    // every rank of a distributed matrix takes part in the exchange, also one that needs no ghosts
    const bool halo = A->distributed;
    const bool has_ghost = A->halo.n_ghost > 0;
    const int64_t unit = 1;
    const int64_t n_units = A->n_rows;
    if (!halo) {
        seg[nseg++] = {0, n_units, false};
    } else {
        // rows [interior_begin, interior_end) touch no ghost column: they run while the halo is
        // in flight, then the boundary strips (variant 3: whole tiles inside the interior).
        BIS_CHECK(bis_halo_exchange_begin(c, A, x));
        const int64_t ib = (A->halo.interior_begin + unit - 1) / unit, ie = A->halo.interior_end / unit;
        if (!has_ghost) {
            seg[nseg++] = {0, n_units, false};
        } else if (ie > ib) {
            seg[nseg++] = {ib, ie - ib, false};
            if (ib > 0) seg[nseg++] = {0, ib, true};
            if (n_units > ie) seg[nseg++] = {ie, n_units - ie, true};
        } else {
            seg[nseg++] = {0, n_units, true};
        }
    }
    bool halo_ended = false;
    for (int i = 0; i < nseg; ++i) {
        if (halo && seg[i].ghost && (i == 0 || !seg[i - 1].ghost)) {
            BIS_CHECK(bis_halo_exchange_end(c, A));
            halo_ended = true;
        }
        int nb = 0;
        ra.finalize = (i == nseg - 1) ? 1 : 0;
        BIS_CHECK(launch_segment(c, A, x, seg[i], epi, ra, &nb));
        ra.block_offset += nb;
    }
    // a rank without ghosts may still SEND (non-symmetric neighbour sets): the main stream must not
    // overwrite x before the NCCL transport's pack on the comm stream has read it
    if (halo && !halo_ended) BIS_CHECK(bis_halo_exchange_end(c, A));
    BIS_CHECK(bis_prof_end(c, BIS_PROF_SPMV));
    if (Epi::NRED > 0) BIS_CHECK(bis_reduce_finish(c, slot_a, slot_b));
    return 0;
}

extern "C" int bis_spmv(bis_context *c, const bis_matrix *A, const double *x, double *y) {
    BIS_REQUIRE(y, "bis_spmv: null y");
    EpiStore e{y};
    return spmv_driver(c, A, x, e, -1, -1);
}

extern "C" int bis_spmv_dot(bis_context *c, const bis_matrix *A, const double *x, double *y,
                            const double *w, int slot_yw, int slot_yy) {
    BIS_REQUIRE(y && w, "bis_spmv_dot: null argument");
    BIS_REQUIRE(slot_yw >= 0 && slot_yw < BIS_NUM_SCALARS && slot_yy < BIS_NUM_SCALARS,
                "bis_spmv_dot: bad slot");
    EpiDot e{y, w};
    return spmv_driver(c, A, x, e, slot_yw, slot_yy);
}

extern "C" int bis_spmv_residual(bis_context *c, const bis_matrix *A, const double *x,
                                 const double *b, double *r, double *tmp, int slot_rr) {
    BIS_REQUIRE(b && r, "bis_spmv_residual: null argument");
    BIS_REQUIRE(slot_rr >= 0 && slot_rr < BIS_NUM_SCALARS, "bis_spmv_residual: bad slot");
    EpiResid e{b, r, tmp};
    return spmv_driver(c, A, x, e, slot_rr, -1);
}

extern "C" int bis_spmv_jacobi(bis_context *c, const bis_matrix *A, const double *D,
                               const double *b, const double *x_old, double *x_new) {
    BIS_REQUIRE(D && b && x_new, "bis_spmv_jacobi: null argument");
    EpiJacobi e{D, b, x_old, x_new};
    return spmv_driver(c, A, x_old, e, -1, -1);
}

extern "C" int bis_spmv_jacobi_residual(bis_context *c, const bis_matrix *A, const double *D, const double *b,
                                        const double *x_old, double *x_new, double *res, int slot_rr) {
    BIS_REQUIRE(D && b && x_new, "bis_spmv_jacobi_residual: null argument");
    BIS_REQUIRE(slot_rr >= 0 && slot_rr < BIS_NUM_SCALARS, "bis_spmv_jacobi_residual: bad scalar slot %d", slot_rr);
    BIS_REQUIRE(x_new != x_old, "bis_spmv_jacobi_residual: the sweep is not an in-place operation");
    EpiJacobiResid e{D, b, x_old, x_new, res};
    return spmv_driver(c, A, x_old, e, slot_rr, -1);
}

extern "C" int bis_spmv_sub(bis_context *c, const bis_matrix *T, const double *x, const double *b,
                            double *out) {
    BIS_REQUIRE(b && out, "bis_spmv_sub: null argument");
    EpiSub e{b, out};
    return spmv_driver(c, T, x, e, -1, -1);
}

// two_stage_gauss_seidel's inner iteration (kernels.hpp:321-331): work_out = -(D_inv . (T work_in)), output += work_out
extern "C" int bis_spmv_two_stage(bis_context *c, const bis_matrix *T, const double *D_inv, const double *work_in,
                                  double *work_out, double *output) {
    BIS_REQUIRE(D_inv && work_out && output, "bis_spmv_two_stage: null argument");
    BIS_REQUIRE(work_in != work_out && work_in != output, "bis_spmv_two_stage: the input vector is read by other rows");
    EpiTwoStage e{D_inv, work_out, output};
    return spmv_driver(c, T, work_in, e, -1, -1);
}

// compute_residual, kernels.hpp:155-162 (tmp is materialised as the reference does)
extern "C" int bis_compute_residual(bis_context *c, const bis_matrix *A, const double *x,
                                    const double *b, double *residual, double *tmp) {
    BIS_REQUIRE(tmp, "bis_compute_residual: null tmp");
    return bis_spmv_residual(c, A, x, b, residual, tmp, BIS_NUM_SCALARS - 2);
}
