// bis_sptrsv.cu -- forward / backward sparse triangular solves
// (native_sptrsv kernels.hpp:54-76, native_bsptrsv kernels.hpp:88-107) and
// apply_preconditioner (kernels.hpp:336-414).
//
// The reference walks the rows strictly in sequence.  The value of a row does
// not depend on the schedule, only on its own summation order, so the rows are
// processed here in LEVEL order (level(r) = 1 + max level of the rows it reads)
// by ONE launch: a thread owns a row, adds its products left to right in
// storage order with unfused multiply/add (bit-identical to the reference's
// scalar loop, SURVEY.md F12), and a warp starts a level once the completion
// counter of the previous level has reached that level's size.  Blocks take
// their chunk of the level-ordered row list from a ticket counter, so a block
// only ever waits for blocks that already run: no co-residency assumption, no
// grid barrier, no deadlock.  The factor is stored a second time in level order
// (LevelSets::d_rp/d_col/d_val) so that consecutive threads stream consecutive
// rows; each thread prefetches its row into registers BEFORE it waits, which
// takes the HBM latency off the level-to-level critical path.
//
// Roofline: HBM for the bytes (12*nnz + 4*n level ids + 4*n row ids +
// sizeof(rp)*n + 24*n for b, D, x), but the run time is bounded below by
// n_levels x (L2 round trip + fence): latency-bound for stencil orderings
// (HPCG-n has 7n-6 levels).
#include "bis_device.cuh"
#include "bis_sptrsv_chain.cuh"
#include "bis_sptrsv_wave.cuh"

#include <algorithm>

#include <cstdlib>

namespace {

constexpr int TRSV_THREADS = 256;
constexpr int TRSV_PF = 16;   // nonzeros prefetched into registers per row

struct TrsvArgs {
    int64_t n_slots;
    const int *slot_row;
    const int *slot_level;
    const int4 *gate;              // per slot: three gate slots + packed distances (nullptr: no staged waiting)
    unsigned int gate_sleep[16];   // ns between polls, by the gate's level distance
    unsigned long long *dbg;       // debug timestamps (4 per row) or nullptr
    unsigned int poll_ns;          // sleep between two polls of the missing operands
    const int64_t *rp;             // level-ordered copy: rows in slot order, operands named by slot
    const int *col;
    const double *val;
    const int *level_size;
    unsigned int *level_done;
    unsigned int *ticket;
    int *errflag;
    double *x;
    const double *D;
    const double *b;
    int post_mul_d;                // store x[row] = D[row] * result (the "tmp <- D tmp" of the SGS preconditioner, kernels.hpp:366-370)
    double *w_clean;               // the working vector of the PREVIOUS solve with this factor: reset to "not ready" here
};

__device__ __forceinline__ unsigned int ld_volatile_u32(const unsigned int *p) {
    return *reinterpret_cast<const volatile unsigned int *>(p);
}

// Comparison variant (opt "trsv_variant" = 2): per-level completion counters.
__global__ void __launch_bounds__(TRSV_THREADS) sptrsv_level_kernel(TrsvArgs a, double *w) {
    __shared__ unsigned int s_chunk;
    if (threadIdx.x == 0) s_chunk = atomicAdd(a.ticket, 1u);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t slot = (int64_t)s_chunk * TRSV_THREADS + threadIdx.x;
    const bool live = slot < a.n_slots;

    int row = 0, lvl = 0x7fffffff;
    int64_t s = 0, e = 0;
    double bb = 0.0, dd = 1.0;
    if (live) {
        row = a.slot_row[slot];
        lvl = a.slot_level[slot];
        s = a.rp[slot];
        e = a.rp[slot + 1];
        bb = a.b[row];
        dd = a.D[row];
    }
    double av[TRSV_PF];
    int cv[TRSV_PF];
#pragma unroll
    for (int j = 0; j < TRSV_PF; ++j) {
        const bool ok = s + j < e;
        av[j] = ok ? __ldcs(a.val + s + j) : 0.0;
        cv[j] = ok ? __ldcs(a.col + s + j) : 0;
    }
    int lv_lo = lvl, lv_hi = live ? lvl : -1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lv_lo = min(lv_lo, __shfl_xor_sync(0xffffffffu, lv_lo, o));
        lv_hi = max(lv_hi, __shfl_xor_sync(0xffffffffu, lv_hi, o));
    }
    for (int lv = lv_lo; lv <= lv_hi; ++lv) {
        if (lv > 0) {
            if (lane == 0) {
                const unsigned int need = (unsigned int)a.level_size[lv - 1];
                long long t0 = clock64();
                unsigned int spins = 0;
                while (ld_volatile_u32(a.level_done + (lv - 1)) < need) {
                    if ((++spins & 1023u) == 0) {
                        if (*reinterpret_cast<volatile int *>(a.errflag)) break;
                        if (clock64() - t0 > 120000000000LL) {   // ~60 s: something is broken
                            atomicExch(a.errflag, 1);
                            break;
                        }
                    }
                }
                __threadfence();   // acquire: order the operand loads after the counter read
            }
            __syncwarp();
        }
        const bool mine = live && lvl == lv;
        if (mine) {
            double sum = 0.0;
#pragma unroll
            for (int j = 0; j < TRSV_PF; ++j)
                if (s + j < e) sum = add_rn(sum, mul_rn(av[j], __ldcg(w + cv[j])));
            for (int64_t k = s + TRSV_PF; k < e; ++k)
                sum = add_rn(sum, mul_rn(a.val[k], __ldcg(w + a.col[k])));
            const double r = div_rn(sub_rn(bb, sum), dd);
            __stcg(w + slot, r);
            a.x[row] = a.post_mul_d ? mul_rn(r, dd) : r;
            __threadfence();   // release: the value is visible before the counter moves
        }
        const unsigned int m = __ballot_sync(0xffffffffu, mine);
        if (lane == 0 && m) atomicAdd(a.level_done + lv, (unsigned int)__popc(m));
    }
}

// ---- default: the value is its own ready flag ("sync-free" in level order) -----------------------
// A row waits only for the rows it actually reads, and what it polls is the value itself: results go
// to a working vector w (in SLOT order) that is pre-filled with a sentinel (a NaN payload the
// arithmetic can never produce); a consumer re-reads w[dep] (8-byte loads are single-copy atomic)
// until it is not the sentinel -- the load that observes readiness also delivers the operand, so one
// hop of the dependency chain costs one store-to-L2 plus one load-from-L2, with no fence and no second
// round trip.  Rows are handed out in level order through the ticket counter, so every dependency
// belongs to an earlier slot, i.e. to a block that is already running (or to an earlier level handled
// by this very warp): no deadlock, no co-residency assumption.  x may alias b (each thread reads its
// b[row] before any x is written and nobody else touches that element).  Summation order per row is
// unchanged: bit-identical results.
//
// What the hop costs was measured (tools/micro/latency.cu, wavefront.cu, tools/trsv_trace.py): 0.28 us
// for a clean L2 store -> poll, but 2.3 us in the first version of this kernel.  Three things made the
// difference, in this order:
//  * every poll touched 32 scattered sectors per operand (w indexed by row): w is now in slot order,
//    the warp's results are one 256-byte store and its operands a few sectors of the previous levels;
//  * lanes left the wait loop one by one and the warp then time-multiplexed a polling path and a
//    computing path: the wait loop is warp-uniform (leave when all rows of the level are ready);
//  * a poll round chained its loads (each predicated on the previous load's result): the loads of a
//    round are predicated on a bit mask and are all in flight together;
// and rows far ahead of the wavefront wait on their "gates" (bis_matrix.cu) with long sleeps instead of
// polling every operand.
constexpr unsigned long long TRSV_SENTINEL = 0xFFF87E5E7E5E7E5EULL;
// watchdog: 60 s WITHOUT PROGRESS (the timer restarts whenever an operand arrives), the rule of the
// factor kernels -- a healthy solve under compute-sanitizer, ncu replay or time-slicing must not trip it
constexpr unsigned long long TRSV_WATCHDOG_NS = 60000000000ull;

__device__ __forceinline__ unsigned long long ld_relaxed_u64(const double *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(256) trsv_fill_sentinel_kernel(int64_t n, double *w) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        reinterpret_cast<unsigned long long *>(w)[i] = TRSV_SENTINEL;
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS) sptrsv_flag_kernel(TrsvArgs a, double *w) {
    __shared__ unsigned int s_chunk;
    if (threadIdx.x == 0) s_chunk = atomicAdd(a.ticket, 1u);
    __syncthreads();
    const int64_t slot = (int64_t)s_chunk * THREADS + threadIdx.x;
    const bool live = slot < a.n_slots;

    int row = 0, lvl = 0x7fffffff;
    int64_t s = 0, e = 0;
    double bb = 0.0, dd = 1.0;
    if (live) {
        row = a.slot_row[slot];
        lvl = a.slot_level[slot];
        s = a.rp[slot];
        e = a.rp[slot + 1];
        bb = a.b[row];
        dd = a.D[row];
        // two working vectors alternate: this solve marks the other one "not ready" for the next solve
        // (nobody reads it any more), so no separate fill launch precedes a solve
        reinterpret_cast<unsigned long long *>(a.w_clean)[slot] = TRSV_SENTINEL;
    }
    // the head of the row is in registers before anything is waited for
    double av[TRSV_PF];
    int cv[TRSV_PF];
#pragma unroll
    for (int j = 0; j < TRSV_PF; ++j) {
        const bool ok = s + j < e;
        av[j] = ok ? __ldcs(a.val + s + j) : 0.0;
        cv[j] = ok ? __ldcs(a.col + s + j) : -1;
    }
    // rows of one warp are consecutive slots, i.e. at most a few consecutive levels; rows of the same
    // level never read one another, so the warp handles its levels one after the other in lockstep
    int lv_lo = lvl, lv_hi = live ? lvl : -1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lv_lo = min(lv_lo, __shfl_xor_sync(0xffffffffu, lv_lo, o));
        lv_hi = max(lv_hi, __shfl_xor_sync(0xffffffffu, lv_hi, o));
    }
    // staged waiting: one gate at a time, oldest first, sleeping in proportion to its distance
    if (a.gate && live) {
        const int4 g = a.gate[slot];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const int gc = i == 0 ? g.x : (i == 1 ? g.y : g.z);
            if (gc < 0) continue;
            const unsigned int ns = a.gate_sleep[(g.w >> (8 * i)) & 15];
            unsigned int spins = 0;
            unsigned long long t_gate = 0;
            while (ld_relaxed_u64(w + gc) == TRSV_SENTINEL) {
                if (ns) __nanosleep(ns);
                if ((++spins & 1023u) == 0) {
                    if (t_gate == 0) t_gate = bis_globaltimer();
                    if (*reinterpret_cast<volatile int *>(a.errflag)) break;
                    if (bis_globaltimer() - t_gate > TRSV_WATCHDOG_NS) {
                        atomicExch(a.errflag, 2);
                        break;
                    }
                }
            }
        }
    }
    __syncwarp();
    // operands: everything already published is taken now; only the missing ones are polled, and the
    // load that finds a value is the load that delivers it (no second round trip)
    unsigned long long xv[TRSV_PF];
#pragma unroll
    for (int j = 0; j < TRSV_PF; ++j) xv[j] = cv[j] >= 0 ? ld_relaxed_u64(w + cv[j]) : 0ull;
    // bit j: operand j has not been seen yet.  The mask, not the loaded values, decides which loads a
    // poll round issues, so that all of them are in flight together.
    unsigned int miss = 0u;
#pragma unroll
    for (int j = 0; j < TRSV_PF; ++j) miss |= (xv[j] == TRSV_SENTINEL ? 1u : 0u) << j;

    for (int lv = lv_lo; lv <= lv_hi; ++lv) {
        const bool mine = live && lvl == lv;
        unsigned long long ts0 = 0, ts1 = 0, ts2 = 0, ts_first = 0, t_wd = 0;
        unsigned int spins = 0;
        bool ok = true;
        if (a.dbg) ts0 = bis_globaltimer();
        // warp-uniform wait: the warp moves on when every row of this level has its operands
        for (;;) {
            if (mine && miss) {
                const unsigned int before = miss;
#pragma unroll
                for (int j = 0; j < TRSV_PF; ++j)
                    if (miss & (1u << j)) xv[j] = ld_relaxed_u64(w + cv[j]);
#pragma unroll
                for (int j = 0; j < TRSV_PF; ++j)
                    if (xv[j] != TRSV_SENTINEL) miss &= ~(1u << j);
                if (miss != before) t_wd = 0;   // progress
            }
            if (__all_sync(0xffffffffu, !mine || miss == 0u)) break;
            if (a.dbg && spins == 0) ts_first = bis_globaltimer();
            if (a.poll_ns) __nanosleep(a.poll_ns);
            bool give_up = false;
            if ((++spins & 4095u) == 0) {
                if (t_wd == 0) t_wd = bis_globaltimer();
                give_up = *reinterpret_cast<volatile int *>(a.errflag) != 0 || bis_globaltimer() - t_wd > TRSV_WATCHDOG_NS;
            }
            if (__any_sync(0xffffffffu, give_up)) {
                atomicExch(a.errflag, 1);
                ok = false;
                break;
            }
        }
        // a warp that gave up publishes nothing: its rows stay "not ready" and their readers give up too
        if (mine && ok) {
            if (a.dbg) ts1 = bis_globaltimer();
            double sum = 0.0;
#pragma unroll
            for (int j = 0; j < TRSV_PF; ++j)
                if (cv[j] >= 0) sum = add_rn(sum, mul_rn(av[j], __longlong_as_double((long long)xv[j])));
            bool tail_ok = true;
            for (int64_t k = s + TRSV_PF; tail_ok && k < e; ++k) {   // rows longer than the register window
                unsigned long long t, t_tail = 0;
                unsigned int sp2 = 0;
                while ((t = ld_relaxed_u64(w + a.col[k])) == TRSV_SENTINEL) {
                    if ((++sp2 & 0xffffu) == 0) {
                        if (t_tail == 0) t_tail = bis_globaltimer();
                        if (*reinterpret_cast<volatile int *>(a.errflag) || bis_globaltimer() - t_tail > TRSV_WATCHDOG_NS) {
                            atomicExch(a.errflag, 1);
                            tail_ok = false;
                            break;
                        }
                    }
                }
                sum = add_rn(sum, mul_rn(a.val[k], __longlong_as_double((long long)t)));
            }
            const double r = div_rn(sub_rn(bb, sum), dd);
            // publish: the value doubles as the flag.  A result that IS the sentinel pattern cannot occur
            // (hardware NaNs are canonical), so readers can never mistake a result for "not ready".
            if (tail_ok) {
                __stcg(w + slot, r);
                a.x[row] = a.post_mul_d ? mul_rn(r, dd) : r;
            }
            if (a.dbg) {
                ts2 = bis_globaltimer();
                a.dbg[4 * (int64_t)row] = ts0;       // the row's level came up in its warp
                a.dbg[4 * (int64_t)row + 1] = ts1;   // all operands in registers
                a.dbg[4 * (int64_t)row + 2] = ts2;   // result published
                // poll rounds that found something missing, and how long the first one took
                a.dbg[4 * (int64_t)row + 3] = (unsigned long long)spins | ((ts_first ? ts_first - ts0 : 0ull) << 32);
            }
        }
        __syncwarp();
    }
}

// Safety-net variant: one launch per level (opt "trsv_variant" = 1).
__global__ void __launch_bounds__(TRSV_THREADS)
sptrsv_one_level_kernel(TrsvArgs a, double *w, int64_t slot_begin, int64_t slot_end) {
    const int64_t slot = slot_begin + (int64_t)blockIdx.x * TRSV_THREADS + threadIdx.x;
    if (slot >= slot_end) return;
    const int row = a.slot_row[slot];
    const int64_t s = a.rp[slot], e = a.rp[slot + 1];
    double sum = 0.0;
    for (int64_t k = s; k < e; ++k) sum = add_rn(sum, mul_rn(a.val[k], __ldcg(w + a.col[k])));
    const double dd = a.D[row];
    const double r = div_rn(sub_rn(a.b[row], sum), dd);
    w[slot] = r;
    a.x[row] = a.post_mul_d ? mul_rn(r, dd) : r;
}

} // namespace

// ---- variant 4: chains (bis_sptrsv_chain.cuh) ---------------------------------------------------------
template <typename RP>
static int chain_build_t(bis_context *c, const bis_matrix *T) {
    ChainFormat &cf = T->lv.chain;
    cf.state = -1;
    const int64_t n = T->n_rows;
    const int upper = T->triangular == 2 ? 1 : 0;
    // record width: the smallest instantiated kernel width that holds the longest row
    const int K = T->max_row <= 4 ? 4 : T->max_row <= 8 ? 8 : T->max_row <= 14 ? 14 : 16;
    if (n < 64 || T->max_row < 1 || T->max_row > chain::KMAX || !T->lv.d_level) return 0;
    cudaStream_t st = c->stream;
    auto pol = thrust::cuda::par.on(st);
    const RP *rp = static_cast<const RP *>(T->d_rp);
    const int grid = bis_blocks_for(n, 256, c->sm_count * 16);
    int *head = nullptr, *cid = nullptr, *chain_start = nullptr, *lmin = nullptr, *pos = nullptr;
    long long *steps = nullptr;
    auto cleanup = [&]() {
        cudaFree(head); cudaFree(cid); cudaFree(chain_start); cudaFree(lmin); cudaFree(pos);
    };
    BIS_CUDA(bis_cuda_malloc(&head, sizeof(int) * (size_t)n));
    BIS_CUDA(bis_cuda_malloc(&cid, sizeof(int) * (size_t)n));
    chain::head_kernel<RP><<<grid, 256, 0, st>>>(n, rp, T->d_col, upper, head);
    BIS_LAUNCH_CHECK(c);
    thrust::inclusive_scan(pol, thrust::device_pointer_cast(head), thrust::device_pointer_cast(head) + n,
                           thrust::device_pointer_cast(cid));
    int n_chains = 0;
    BIS_CUDA(cudaMemcpyAsync(&n_chains, cid + (n - 1), sizeof(int), cudaMemcpyDeviceToHost, st));
    BIS_CUDA(cudaStreamSynchronize(st));
    const int n_groups = (n_chains + 31) / 32;
    BIS_CUDA(bis_cuda_malloc(&chain_start, sizeof(int) * ((size_t)n_chains + 1)));
    BIS_CUDA(bis_cuda_malloc(&lmin, sizeof(int) * (size_t)n_groups));
    BIS_CUDA(bis_cuda_malloc(&steps, sizeof(long long) * ((size_t)n_groups + 1)));
    chain::chain_start_kernel<<<grid, 256, 0, st>>>(n, head, cid, chain_start, n_chains);
    BIS_LAUNCH_CHECK(c);
    BIS_CUDA(cudaMemsetAsync(steps, 0, sizeof(long long) * ((size_t)n_groups + 1), st));
    chain::group_steps_kernel<<<bis_blocks_for(n_groups, 128, c->sm_count * 8), 128, 0, st>>>(
        n_groups, n_chains, n, upper, chain_start, T->lv.d_level, lmin, steps);
    BIS_LAUNCH_CHECK(c);
    thrust::exclusive_scan(pol, thrust::device_pointer_cast(steps), thrust::device_pointer_cast(steps) + n_groups + 1,
                           thrust::device_pointer_cast(steps));
    long long n_recs = 0;
    BIS_CUDA(cudaMemcpyAsync(&n_recs, steps + n_groups, sizeof(long long), cudaMemcpyDeviceToHost, st));
    BIS_CUDA(cudaStreamSynchronize(st));
    // idle lane-steps are padding: give up when the chains of a warp are too unlike (or too short) to be
    // worth it, and when positions would not fit 31 bits
    if (n_recs * 32 > (long long)(2.5 * (double)n) || n_recs * 32 >= (1ll << 31)) {
        cleanup();
        cudaFree(steps);
        return 0;
    }
    const size_t rb = chain::rec_bytes(K);
    unsigned char *recs = nullptr;
    double *w = nullptr;
    BIS_CUDA(bis_cuda_malloc(&recs, rb * (size_t)n_recs));
    BIS_CUDA(bis_cuda_malloc(&w, sizeof(double) * 32 * (size_t)n_recs));
    BIS_CUDA(bis_cuda_malloc(&pos, sizeof(int) * (size_t)n));
    chain::rec_init_kernel<<<c->sm_count * 16, 256, 0, st>>>(n_recs, K, recs);
    BIS_LAUNCH_CHECK(c);
    chain::pos_kernel<<<grid, 256, 0, st>>>(n, upper, cid, T->lv.d_level, lmin, steps, pos);
    BIS_LAUNCH_CHECK(c);
    chain::rec_fill_kernel<RP><<<grid, 256, 0, st>>>(n, rp, T->d_col, T->d_val, upper, K, cid, T->lv.d_level, lmin, pos, recs);
    BIS_LAUNCH_CHECK(c);
    BIS_CUDA(cudaStreamSynchronize(st));
    cleanup();
    cf.K = K;
    cf.n_groups = n_groups;
    cf.n_recs = n_recs;
    cf.d_recs = recs;
    cf.d_slice_off = steps;
    cf.d_w = w;
    cf.state = 1;
    return 0;
}

static int chain_solve(bis_context *c, const bis_matrix *T, double *x, const double *D, const double *b) {
    const ChainFormat &cf = T->lv.chain;
    chain::Args a;
    a.n_groups = cf.n_groups;
    a.K = cf.K;
    a.recs = cf.d_recs;
    a.slice_off = cf.d_slice_off;
    a.ticket = T->lv.d_ticket;
    a.errflag = c->d_errflag;
    a.x = x;
    a.D = D;
    a.b = b;
    const size_t per_warp = chain::NST * chain::rec_bytes(cf.K) + 32 * 8 * sizeof(double) + 64;
    const size_t smem = per_warp * chain::WARPS;
    void (*kern)(chain::Args, double *) = cf.K == 4 ? chain::chain_kernel<4> : cf.K == 8 ? chain::chain_kernel<8>
                                           : cf.K == 14 ? chain::chain_kernel<14> : chain::chain_kernel<16>;
    BIS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    BIS_CUDA(cudaMemsetAsync(T->lv.d_ticket, 0, sizeof(unsigned int), c->stream));
    chain::fill_sentinel_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(32 * cf.n_recs, cf.d_w);
    BIS_LAUNCH_CHECK(c);
    const int blocks = (cf.n_groups + chain::WARPS - 1) / chain::WARPS;
    kern<<<blocks, chain::WARPS * 32, smem, c->stream>>>(a, cf.d_w);
    BIS_LAUNCH_CHECK(c);
    return 0;
}

// ---- variant 5: stencil wavefront (bis_sptrsv_wave.cuh) ------------------------------------------------
namespace {

template <typename RP>
int wave_try_grid(bis_context *c, const bis_matrix *T, int nx, int ny, int nz, bool *ok) {
    *ok = false;
    const int64_t n = T->n_rows;
    if (nx < 1 || ny < 1 || nz < 1 || (int64_t)nx * ny * nz != n) return 0;
    if (nx < 4 && n > 64) return 0;               // the lane skew assumes lines, not dots
    if ((ny + 31) / 32 > wave::MAX_WARPS) return 0;  // a plane must fit one CTA (its lines share the CTA's rings)
    wave::Grid g;
    g.nx = nx; g.ny = ny; g.nz = nz;
    g.W = (ny + 31) / 32;
    g.S = nx + 62;
    g.n = n;
    g.upper = T->triangular == 2 ? 1 : 0;
    int *d_status = nullptr;
    BIS_CUDA(bis_cuda_malloc(&d_status, sizeof(int)));
    BIS_CUDA(cudaMemsetAsync(d_status, 0, sizeof(int), c->stream));
    const int grid = bis_blocks_for(n, 256, c->sm_count * 16);
    wave::validate_kernel<RP><<<grid, 256, 0, c->stream>>>(g, static_cast<const RP *>(T->d_rp), T->d_col, d_status);
    BIS_LAUNCH_CHECK(c);
    int status = 0;
    BIS_CUDA(cudaMemcpyAsync(&status, d_status, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(d_status);
    if (status != 0) return 0;
    WaveFormat &wf = T->lv.wave;
    wf.nx = nx; wf.ny = ny; wf.nz = nz; wf.W = g.W; wf.S = g.S;
    wf.n_groups = wave::n_groups(g);
    *ok = true;
    return 0;
}

// distinct |row - col| of the factor, ascending (empty when there are more than a stencil has)
template <typename RP>
int wave_offsets(bis_context *c, const bis_matrix *T, std::vector<int> *out) {
    out->clear();
    int *d_tab = nullptr;
    const size_t bytes = sizeof(int) * (wave::OFFS_CAP + 2);
    BIS_CUDA(bis_cuda_malloc(&d_tab, bytes));
    BIS_CUDA(cudaMemsetAsync(d_tab, 0, bytes, c->stream));
    wave::offsets_kernel<RP><<<bis_blocks_for(T->n_rows, 256, c->sm_count * 8), 256, 0, c->stream>>>(
        T->n_rows, static_cast<const RP *>(T->d_rp), T->d_col, d_tab);
    BIS_LAUNCH_CHECK(c);
    int tab[wave::OFFS_CAP + 2];
    BIS_CUDA(cudaMemcpyAsync(tab, d_tab, bytes, cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    cudaFree(d_tab);
    if (tab[wave::OFFS_CAP + 1] != 0 || tab[0] > 13) return 0;
    for (int i = 0; i < tab[0]; ++i) out->push_back(tab[1 + i]);
    std::sort(out->begin(), out->end());
    return 0;
}

template <typename RP>
int wave_build_t(bis_context *c, const bis_matrix *T) {
    WaveFormat &wf = T->lv.wave;
    wf.state = -1;
    const int64_t n = T->n_rows;
    if (n < 32 || T->nnz == 0 || T->max_row > wave::K || T->triangular == 0) return 0;
    bool ok = false;
    if (T->grid_nx > 0) {
        BIS_CHECK(wave_try_grid<RP>(c, T, (int)T->grid_nx, (int)T->grid_ny, (int)T->grid_nz, &ok));
    } else {
        // no hint (an uploaded factor): the grid is read off the distinct offsets 1, nx-1..nx+1, P-nx-1..P+nx+1
        std::vector<int> offs;
        BIS_CHECK(wave_offsets<RP>(c, T, &offs));
        std::vector<int> nx_c, p_c;
        if (!offs.empty() && offs[0] == 1) {
            size_t i = 1;
            if (i < offs.size()) {
                const int a = offs[i];
                for (int cand : {a + 1, a}) nx_c.push_back(cand);
            } else {
                nx_c.push_back((int)n);          // a single chain
            }
        } else if (!offs.empty()) {
            nx_c.push_back(offs[0]);             // no x-coupling at all
            nx_c.push_back(offs[0] + 1);
        }
        for (int nx : nx_c) {
            if (ok) break;
            if (nx < 1 || n % nx != 0) continue;
            p_c.clear();
            for (int o : offs)
                if (o > nx + 1) {
                    for (int cand : {o, o + 1, o + nx - 1, o + nx, o + nx + 1}) p_c.push_back(cand);
                    break;
                }
            p_c.push_back((int)n);               // a single plane
            for (int P : p_c) {
                if (P < nx || P % nx != 0 || n % P != 0) continue;
                BIS_CHECK(wave_try_grid<RP>(c, T, nx, P / nx, (int)(n / P), &ok));
                if (ok) break;
            }
        }
    }
    if (!ok) return 0;
    if (c->opt_trsv_variant != 5) {
        // automatic choice (the level analysis has run): the wavefront pays ~4 us per PLANE (hand-over from plane to
        // plane: 2.3 us at four blocks per plane, 4.3 us at eight, with clusters of eight planes) plus ~0.5 us per
        // step of one plane, the dataflow solve ~1.3 us per LEVEL (measured on B200, profiles/r02_wave_*, r02b_wave_*).
        // 27-point factors have 4 levels per plane and win; 7-point factors have 1 and do not.
        const double est_wave = 4.0 * wf.nz + 0.5 * (wf.nx + 2.0 * wf.ny + 64.0 * (wf.W - 1));
        const double est_flow = 1.3 * T->lv.n_levels;
        if (!T->lv.built || est_wave >= est_flow) {
            wf.state = -2;      // a stencil, but not worth it
            return 0;
        }
    }
    // records (zeros where a neighbour does not exist) and the two working vectors, both "not ready"
    const size_t rec_doubles = (size_t)wf.n_groups * wf.S * wave::REC_DOUBLES;
    const size_t w_doubles = (size_t)wf.n_groups * wf.S * 32;
    size_t fr = 0, tot = 0;
    if (cudaMemGetInfo(&fr, &tot) == cudaSuccess && (rec_doubles + 2 * w_doubles) * 8 + ((size_t)1 << 30) > fr) {
        bis_vector_cache_release_all();
        if (cudaMemGetInfo(&fr, &tot) == cudaSuccess && (rec_doubles + 2 * w_doubles) * 8 + ((size_t)1 << 30) > fr) return 0;   // no room: dataflow solve
    }
    BIS_CUDA(bis_cuda_malloc(&wf.d_rec, rec_doubles * 8));
    BIS_CUDA(bis_cuda_malloc(&wf.d_w[0], w_doubles * 8));
    BIS_CUDA(bis_cuda_malloc(&wf.d_w[1], w_doubles * 8));
    BIS_CUDA(bis_cuda_malloc(&wf.d_ticket, sizeof(unsigned int)));
    BIS_CUDA(cudaMemsetAsync(wf.d_rec, 0, rec_doubles * 8, c->stream));
    wave::Grid g;
    g.nx = wf.nx; g.ny = wf.ny; g.nz = wf.nz; g.W = wf.W; g.S = wf.S; g.n = n; g.upper = T->triangular == 2 ? 1 : 0;
    const int grid = bis_blocks_for(n, 256, c->sm_count * 16);
    wave::fill_kernel<RP><<<grid, 256, 0, c->stream>>>(g, static_cast<const RP *>(T->d_rp), T->d_col, T->d_val, wf.d_rec);
    BIS_LAUNCH_CHECK(c);
    for (int i = 0; i < 2; ++i) {
        wave::fill_u64_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>((long long)w_doubles, reinterpret_cast<unsigned long long *>(wf.d_w[i]), wave::SENT);
        BIS_LAUNCH_CHECK(c);
        wf.w_clean[i] = 1;
    }
    wf.w_epoch = c->graph_epoch;
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    wf.state = 1;
    return 0;
}

int wave_solve(bis_context *c, const bis_matrix *T, double *x, const double *D, const double *b, int post_mul_d) {
    WaveFormat &wf = T->lv.wave;
    wave::Args a;
    a.g.nx = wf.nx; a.g.ny = wf.ny; a.g.nz = wf.nz; a.g.W = wf.W; a.g.S = wf.S; a.g.n = T->n_rows;
    a.g.upper = T->triangular == 2 ? 1 : 0;
    a.rec = wf.d_rec;
    a.ticket = wf.d_ticket;
    a.errflag = c->d_errflag;
    a.x = x; a.D = D; a.b = b;
    a.post_mul_d = post_mul_d;
#ifdef BIS_PERF_DEBUG
    a.dbg = c->opt_wave_debug;
    a.stamps = nullptr;
    const char *stamp_file = (c->opt_wave_debug & 64) ? getenv("BIS_WAVE_STAMPS") : nullptr;
    if (stamp_file) BIS_CUDA(bis_cuda_malloc(&a.stamps, sizeof(unsigned long long) * (2 * (size_t)wf.nz + 64)));
#endif
    const size_t smem = wave::smem_bytes(wf.W);
    const void *fn = a.g.upper ? reinterpret_cast<const void *>(wave::wave_kernel<true>) : reinterpret_cast<const void *>(wave::wave_kernel<false>);
    BIS_CHECK(bis_ensure_dynamic_smem(c, fn, smem));
    // consecutive planes run in the CTAs of one thread-block cluster and hand their values over through distributed
    // shared memory (option wave_cluster: planes per cluster, 1 = everything through L2): the largest size <= the
    // option of which at least one cluster fits the device
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3((unsigned)((wf.W * wave::PH * 32 + 32)));
    cfg.dynamicSmemBytes = smem;
    cfg.stream = c->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int cl = c->opt_wave_cluster < 1 ? 1 : (c->opt_wave_cluster > 16 ? 16 : c->opt_wave_cluster);
    if (cl > 8 && cudaFuncSetAttribute(fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) {
        cudaGetLastError();
        cl = 8;
    }
    while (cl > 1 && (cl & (cl - 1))) --cl;
    while (cl > 1 && cl > wf.nz) cl >>= 1;
    int n_clusters = 0;
    for (; cl > 1; cl >>= 1) {
        if (wf.cluster_fit[cl] < 0) {       // asked once per factor and size
            attr[0].val.clusterDim.x = (unsigned)cl; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
            cfg.gridDim = dim3((unsigned)(cl * c->sm_count));
            int fit = 0;
            if (cudaOccupancyMaxActiveClusters(&fit, fn, &cfg) != cudaSuccess) {
                cudaGetLastError();
                fit = 0;
            }
            wf.cluster_fit[cl] = fit;
        }
        if (wf.cluster_fit[cl] > 0) {
            n_clusters = wf.cluster_fit[cl];
            break;
        }
    }
    if (wf.w_cluster != cl) {      // which planes leave a copy in the working vectors depends on the cluster size
        wf.w_clean[0] = wf.w_clean[1] = 0;
        wf.w_cluster = cl;
    }
    if (wf.w_epoch != c->graph_epoch || c->capturing) {   // a graph replay may have used either vector since
        wf.w_clean[0] = wf.w_clean[1] = 0;
        wf.w_epoch = c->graph_epoch;
    }
    int p = wf.w_clean[0] ? 0 : (wf.w_clean[1] ? 1 : -1);
#ifdef BIS_PERF_DEBUG
    static bool dbg128_armed = false;   // experiment below: the first such solve fills d_w[0], the later ones only read it
    if ((c->opt_wave_debug & 128) && dbg128_armed) p = 0;
    if (c->opt_wave_debug & 128) dbg128_armed = true;
#endif
    if (p < 0) {
        wave::fill_u64_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>((long long)wf.n_groups * wf.S * 32,
                                                                      reinterpret_cast<unsigned long long *>(wf.d_w[0]), wave::SENT);
        BIS_LAUNCH_CHECK(c);
        p = 0;
    }
    a.w = wf.d_w[p];
    a.w_clean = wf.d_w[1 - p];
    wf.w_clean[p] = 0;
    wf.w_clean[1 - p] = c->capturing ? 0 : 1;
#ifdef BIS_PERF_DEBUG
    if (c->opt_wave_debug & 128) {   // experiment: read the values the PREVIOUS identical solve left (nobody waits)
        a.w = wf.d_w[0];
        a.w_clean = wf.d_w[1];
        wf.w_clean[0] = wf.w_clean[1] = 0;
    }
#endif
    BIS_CUDA(cudaMemsetAsync(wf.d_ticket, 0, sizeof(unsigned int), c->stream));
    // one CTA per plane in flight, all of a plane's 32-line blocks in it (two warps each)
    a.backoff_ns = cl > 1 ? (unsigned int)c->opt_wave_backoff_ns : 0u;
    if (cl > 1) {
        const int need = (wf.nz + cl - 1) / cl;
        if (n_clusters > need) n_clusters = need;
        attr[0].val.clusterDim.x = (unsigned)cl; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.gridDim = dim3((unsigned)(n_clusters * cl));
        void *kargs[1] = {&a};
        BIS_CUDA(cudaLaunchKernelExC(&cfg, fn, kargs));
    } else {
        int blocks = c->sm_count;
        if (blocks > wf.nz) blocks = wf.nz;
        if (a.g.upper) wave::wave_kernel<true><<<blocks, (wf.W * wave::PH * 32 + 32), smem, c->stream>>>(a);
        else wave::wave_kernel<false><<<blocks, (wf.W * wave::PH * 32 + 32), smem, c->stream>>>(a);
    }
    c->wave_cluster_used = cl;
    if (getenv("BIS_WAVE_VERBOSE")) fprintf(stderr, "[bis] wavefront: %d planes per cluster, %d clusters, %d threads, %zu bytes of shared memory per CTA\n", cl, n_clusters, (wf.W * wave::PH * 32 + 32), smem);
    BIS_LAUNCH_CHECK(c);
#ifdef BIS_PERF_DEBUG
    if (a.stamps) {
        std::vector<unsigned long long> h(2 * (size_t)wf.nz + 64);
        BIS_CUDA(cudaMemcpyAsync(h.data(), a.stamps, sizeof(unsigned long long) * h.size(), cudaMemcpyDeviceToHost, c->stream));
        BIS_CUDA(cudaStreamSynchronize(c->stream));
        if (FILE *f = fopen(stamp_file, "wb")) {
            fwrite(h.data(), sizeof(unsigned long long), h.size(), f);
            fclose(f);
        }
        cudaFree(a.stamps);
    }
#endif
    return 0;
}

} // namespace

int bis_wave_build(bis_context *c, const bis_matrix *T) {
    if (T->lv.wave.state != 0) return 0;
    if (T->crs_released) {      // nothing to build the records from any more
        T->lv.wave.state = -1;
        return 0;
    }
    BIS_CUDA(cudaSetDevice(c->device));
    if (T->rp_bytes == 8) return wave_build_t<int64_t>(c, T);
    return wave_build_t<int32_t>(c, T);
}

// sleeps of the dataflow solves: per gate level distance, and between two polls of the missing operands
static void trsv_wait_params(const bis_context *c, unsigned int gate_sleep[16], unsigned int *poll_ns) {
    const int *sl = c->opt_trsv_sleep;
    for (int d = 0; d < 16; ++d)
        gate_sleep[d] = (unsigned int)(d <= 1 ? sl[0] : d == 2 ? sl[1] : d == 3 ? sl[2] : d < 6 ? sl[3] : 2 * sl[3]);
    *poll_ns = c->opt_trsv_poll_ns > 0 ? (unsigned int)c->opt_trsv_poll_ns : (c->opt_trsv_poll_ns < 0 ? 0u : 20u);   // < 0: spin without sleeping
}

static int trsv_solve(bis_context *c, const bis_matrix *T, double *x, const double *D,
                      const double *b, int want_kind, int post_mul_d = 0) {
    BIS_REQUIRE(c && T && x && D && b, "sptrsv: null argument");
    BIS_REQUIRE(T->triangular == want_kind,
                "sptrsv: matrix is not the %s strictly-triangular factor this call needs",
                want_kind == 1 ? "lower" : "upper");
    BIS_REQUIRE(!T->distributed, "sptrsv: triangular sweeps do not shard (single-GPU only)");
    BisNvtxRange nvtx_range(want_kind == 1 ? "sptrsv" : "backwards-sptrsv");
    BIS_CUDA(cudaSetDevice(c->device));
    LevelSets &lv = T->lv;
    if (T->n_rows == 0) return 0;
    if (c->opt_trsv_variant == 5 && (lv.wave.state == 0 || lv.wave.state == -2)) {   // forced after the factor was made
        lv.wave.state = 0;
        BIS_CHECK(bis_wave_build(c, T));
    }
    if ((c->opt_trsv_variant == 5 || c->opt_trsv_variant == 0) && lv.wave.state == 1) {
        BIS_CHECK(bis_prof_begin(c, BIS_PROF_SPTRSV));
        BIS_CHECK(wave_solve(c, T, x, D, b, post_mul_d));
        c->wave_solves++;
        return bis_prof_end(c, BIS_PROF_SPTRSV);
    }
    BIS_REQUIRE(c->opt_trsv_variant != 5, "trsv_variant=5 forced, but the factor is not a (<= 27-point) stencil in natural ordering");
    BIS_CHECK(bis_ensure_levels(c, T));
    TrsvArgs a;
    a.n_slots = lv.n_slots;
    a.slot_row = lv.d_slot_row;
    a.slot_level = lv.d_slot_level;
    a.gate = c->opt_trsv_gates ? reinterpret_cast<const int4 *>(lv.d_slot_gate) : nullptr;
    trsv_wait_params(c, a.gate_sleep, &a.poll_ns);
    a.rp = lv.d_rp;
    a.col = lv.d_col;
    a.val = lv.d_val;
    a.level_size = lv.d_level_size;
    a.level_done = lv.d_level_done;
    a.ticket = lv.d_ticket;
    a.errflag = c->d_errflag;
    a.dbg = nullptr;
    const char *dbg_file = c->opt_trsv_debug ? getenv("BIS_TRSV_DEBUG_FILE") : nullptr;
    if (dbg_file) BIS_CUDA(bis_cuda_malloc(&a.dbg, sizeof(unsigned long long) * 4 * (size_t)lv.n_slots));
    a.x = x;
    a.D = D;
    a.b = b;
    a.post_mul_d = post_mul_d;
    a.w_clean = nullptr;
    if (c->opt_trsv_variant == 4 && T->lv.chain.state == 0 && !T->crs_released) {
        if (T->rp_bytes == 8) BIS_CHECK(chain_build_t<int64_t>(c, T));
        else BIS_CHECK(chain_build_t<int32_t>(c, T));
    }
    BIS_CHECK(bis_prof_begin(c, BIS_PROF_SPTRSV));
    if (c->opt_trsv_variant == 4 && T->lv.chain.state == 1) {
        BIS_CHECK(chain_solve(c, T, x, D, b));
        c->chain_solves++;
        if (post_mul_d) BIS_CHECK(bis_elemwise_mult_vectors(c, x, x, D, T->n_rows, 1.0));
        return bis_prof_end(c, BIS_PROF_SPTRSV);
    }
    if (c->opt_trsv_variant == 1 || c->opt_trsv_variant == 2) lv.w_clean[0] = 0;   // they leave results in d_w
    if (c->opt_trsv_variant == 1) {
        const std::vector<int64_t> &ls = lv.level_start;
        for (int l = 0; l < lv.n_levels; ++l) {
            int64_t cnt = ls[l + 1] - ls[l];
            int blocks = (int)((cnt + TRSV_THREADS - 1) / TRSV_THREADS);
            sptrsv_one_level_kernel<<<blocks, TRSV_THREADS, 0, c->stream>>>(a, lv.d_w, ls[l], ls[l + 1]);
            BIS_LAUNCH_CHECK(c);
        }
        return bis_prof_end(c, BIS_PROF_SPTRSV);
    }
    const int64_t blocks = (lv.n_slots + TRSV_THREADS - 1) / TRSV_THREADS;
    BIS_CUDA(cudaMemsetAsync(lv.d_ticket, 0, sizeof(unsigned int), c->stream));
    if (c->opt_trsv_variant != 2) {
        // the working vector of this solve is clean (filled at build time, or by the previous solve)
        if (lv.w_epoch != c->graph_epoch || c->capturing) {   // a graph replay may have used either vector since
            lv.w_clean[0] = lv.w_clean[1] = 0;
            lv.w_epoch = c->graph_epoch;
        }
        int p = lv.w_clean[0] ? 0 : (lv.w_clean[1] ? 1 : -1);
        if (p < 0) {   // neither is known to be clean: inside a graph (fixed pointers), after one, or after another variant
            trsv_fill_sentinel_kernel<<<bis_blocks_for(lv.n_slots, 1024, c->sm_count * 8), 256, 0, c->stream>>>(lv.n_slots, lv.d_w);
            BIS_LAUNCH_CHECK(c);
            p = 0;
        }
        double *w_use = p ? lv.d_w2 : lv.d_w;
        a.w_clean = p ? lv.d_w : lv.d_w2;
        lv.w_clean[p] = 0;
        lv.w_clean[1 - p] = c->capturing ? 0 : 1;
        // rows per block (opt "trsv_block"): a block retires when its last row is done, so smaller blocks
        // hand their registers to rows further down the list sooner
        const int tb = c->opt_trsv_block;
        if (tb == 64)
            sptrsv_flag_kernel<64><<<(unsigned int)((lv.n_slots + 63) / 64), 64, 0, c->stream>>>(a, w_use);
        else if (tb == 128)
            sptrsv_flag_kernel<128><<<(unsigned int)((lv.n_slots + 127) / 128), 128, 0, c->stream>>>(a, w_use);
        else
            sptrsv_flag_kernel<256><<<(unsigned int)blocks, 256, 0, c->stream>>>(a, w_use);
        BIS_LAUNCH_CHECK(c);
        if (a.dbg) {   // debug aid (tools/trsv_trace.py): per-row timestamps of the last solve
            std::vector<unsigned long long> h(4 * (size_t)lv.n_slots);
            BIS_CUDA(cudaMemcpyAsync(h.data(), a.dbg, sizeof(unsigned long long) * h.size(), cudaMemcpyDeviceToHost, c->stream));
            BIS_CUDA(cudaStreamSynchronize(c->stream));
            if (FILE *f = fopen(dbg_file, "wb")) {
                fwrite(h.data(), sizeof(unsigned long long), h.size(), f);
                fclose(f);
            }
            cudaFree(a.dbg);
        }
        return bis_prof_end(c, BIS_PROF_SPTRSV);
    }
    // variant 2: per-level completion counters (kept for comparison)
    BIS_CUDA(cudaMemsetAsync(lv.d_level_done, 0, sizeof(unsigned int) * (size_t)lv.n_levels, c->stream));
    sptrsv_level_kernel<<<(unsigned int)blocks, TRSV_THREADS, 0, c->stream>>>(a, lv.d_w);
    BIS_LAUNCH_CHECK(c);
    return bis_prof_end(c, BIS_PROF_SPTRSV);
}

extern "C" int bis_sptrsv(bis_context *c, const bis_matrix *L, double *x, const double *D,
                          const double *b) {
    return trsv_solve(c, L, x, D, b, 1);
}
extern "C" int bis_bsptrsv(bis_context *c, const bis_matrix *U, double *x, const double *D,
                           const double *b) {
    return trsv_solve(c, U, x, D, b, 2);
}

// ---- several right-hand sides (bis_block_sptrsv / bis_block_bsptrsv) -----------------------------------
// The dataflow solve above with k columns carried through every dependency: the same level-ordered copy, the same
// ticket hand-out in slot order, the same "the value is its own ready flag" protocol, on a working array of
// n_slots x k doubles (element (slot, j) at slot*k + j).  A row is served by TPR threads (1, 2, 4, 8 for k <= 2, 4, 8,
// 16); each owns CW <= 2 consecutive columns and polls and publishes only those of them that are active.  The operands
// of a window of PF = 16 nonzeros are polled together, warp-uniformly, and added in storage order; a row longer than
// the window takes further windows, so the sum is that of the single-vector kernel for every column.  Two columns per
// thread keep a whole HPCG factor row (13 nonzeros) in one window: with four columns per thread and an 8-nonzero
// window (what the registers allow) the solve took 6.5 us per level at k = 4..16 against 1.7 us at k = 2 (HPCG-128).
namespace {

template <int K> struct BtrsvShape {
    static constexpr int TPR = K <= 2 ? 1 : (K <= 4 ? 2 : (K <= 8 ? 4 : 8));   // threads per row
    static constexpr int CW = (K + TPR - 1) / TPR;                              // columns per thread (<= 2)
    static constexpr int PF = 16;                                               // nonzeros per window: PF * CW <= 32 poll bits
    static constexpr int ROWS = 256 / TPR;                      // rows per block
};

struct BtrsvArgs {
    int64_t n_slots;
    const int *slot_row;
    const int *slot_level;
    const int4 *gate;
    unsigned int gate_sleep[16];
    unsigned int poll_ns;
    const int64_t *rp;
    const int *col;
    const double *val;
    unsigned int *ticket;
    int *errflag;
    double *X;
    const double *D;
    const double *B;
    const double *active;   // [k] flags or nullptr
    double *w_clean;        // the other working array: reset to "not ready" in [0, n_slots*k)
};

template <int K>
__global__ void __launch_bounds__(256, 1) block_sptrsv_kernel(BtrsvArgs a, double *wk) {
    using S = BtrsvShape<K>;
    constexpr int CW = S::CW, PF = S::PF;
    __shared__ unsigned int s_chunk;
    if (threadIdx.x == 0) s_chunk = atomicAdd(a.ticket, 1u);
    __syncthreads();
    const int64_t slot = (int64_t)s_chunk * S::ROWS + threadIdx.x / S::TPR;
    const int c0 = ((int)threadIdx.x % S::TPR) * CW;
    const bool live = slot < a.n_slots;

    unsigned int act = 0u;   // bit w: column c0 + w exists and is active
#pragma unroll
    for (int w = 0; w < CW; ++w)
        if (c0 + w < K && (a.active == nullptr || a.active[c0 + w] != 0.0)) act |= 1u << w;
    int row = 0, lvl = 0x7fffffff;
    int64_t s = 0, e = 0;
    double bb[CW], dd = 1.0;
#pragma unroll
    for (int w = 0; w < CW; ++w) bb[w] = 0.0;
    if (live) {
        row = a.slot_row[slot];
        lvl = a.slot_level[slot];
        s = a.rp[slot];
        e = a.rp[slot + 1];
        dd = a.D[row];
#pragma unroll
        for (int w = 0; w < CW; ++w) {
            if (act >> w & 1u) bb[w] = a.B[(int64_t)row * K + c0 + w];
            if (c0 + w < K) reinterpret_cast<unsigned long long *>(a.w_clean)[slot * K + c0 + w] = TRSV_SENTINEL;
        }
    } else {
        act = 0u;
    }
    // the head of the row is in registers before anything is waited for
    double av[PF];
    int cv[PF];
#pragma unroll
    for (int j = 0; j < PF; ++j) {
        const bool ok = act && s + j < e;
        av[j] = ok ? __ldcs(a.val + s + j) : 0.0;
        cv[j] = ok ? __ldcs(a.col + s + j) : -1;
    }
    int lv_lo = lvl, lv_hi = live ? lvl : -1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lv_lo = min(lv_lo, __shfl_xor_sync(0xffffffffu, lv_lo, o));
        lv_hi = max(lv_hi, __shfl_xor_sync(0xffffffffu, lv_hi, o));
    }
    // staged waiting on the gates, through the first active column this thread owns
    if (a.gate && act) {
        const int wg = __ffs(act) - 1;
        const int4 g = a.gate[slot];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const int gc = i == 0 ? g.x : (i == 1 ? g.y : g.z);
            if (gc < 0) continue;
            const unsigned int ns = a.gate_sleep[(g.w >> (8 * i)) & 15];
            unsigned int spins = 0;
            unsigned long long t_gate = 0;
            while (ld_relaxed_u64(wk + (int64_t)gc * K + c0 + wg) == TRSV_SENTINEL) {
                if (ns) __nanosleep(ns);
                if ((++spins & 1023u) == 0) {
                    if (t_gate == 0) t_gate = bis_globaltimer();
                    if (*reinterpret_cast<volatile int *>(a.errflag)) break;
                    if (bis_globaltimer() - t_gate > TRSV_WATCHDOG_NS) {
                        atomicExch(a.errflag, 2);
                        break;
                    }
                }
            }
        }
    }
    __syncwarp();
    // operands: everything already published is taken now; operand (j, w) is bit j*CW + w of the poll mask
    unsigned long long xv[PF][CW];
    unsigned int miss = 0u;
    auto take_window = [&]() {
        miss = 0u;
#pragma unroll
        for (int j = 0; j < PF; ++j)
#pragma unroll
            for (int w = 0; w < CW; ++w) {
                const bool use = cv[j] >= 0 && (act >> w & 1u);
                xv[j][w] = use ? ld_relaxed_u64(wk + (int64_t)cv[j] * K + c0 + w) : 0ull;
                if (use && xv[j][w] == TRSV_SENTINEL) miss |= 1u << (j * CW + w);
            }
    };
    take_window();

    for (int lv = lv_lo; lv <= lv_hi; ++lv) {
        const bool mine = act && lvl == lv;
        const int nwin = mine ? (int)((e - s + PF - 1) / PF) : 0;
        const int nwin_max = __reduce_max_sync(0xffffffffu, (unsigned)nwin);
        double sum[CW];
#pragma unroll
        for (int w = 0; w < CW; ++w) sum[w] = 0.0;
        bool ok = true;
        for (int win = 0; win < nwin_max && ok; ++win) {
            if (win > 0 && mine && win < nwin) {   // the next window of a long row
                const int64_t b0 = s + (int64_t)win * PF;
#pragma unroll
                for (int j = 0; j < PF; ++j) {
                    const bool in = b0 + j < e;
                    av[j] = in ? a.val[b0 + j] : 0.0;
                    cv[j] = in ? a.col[b0 + j] : -1;
                }
                take_window();
            }
            const bool here = mine && win < nwin;
            unsigned long long t_wd = 0;
            unsigned int spins = 0;
            // warp-uniform wait: the warp moves on when every row of this level has the operands of this window
            for (;;) {
                if (here && miss) {
                    const unsigned int before = miss;
#pragma unroll
                    for (int j = 0; j < PF; ++j)
#pragma unroll
                        for (int w = 0; w < CW; ++w)
                            if (miss & (1u << (j * CW + w))) xv[j][w] = ld_relaxed_u64(wk + (int64_t)cv[j] * K + c0 + w);
#pragma unroll
                    for (int j = 0; j < PF; ++j)
#pragma unroll
                        for (int w = 0; w < CW; ++w)
                            if (xv[j][w] != TRSV_SENTINEL) miss &= ~(1u << (j * CW + w));
                    if (miss != before) t_wd = 0;   // progress
                }
                if (__all_sync(0xffffffffu, !here || miss == 0u)) break;
                if (a.poll_ns) __nanosleep(a.poll_ns);
                bool give_up = false;
                if ((++spins & 4095u) == 0) {
                    if (t_wd == 0) t_wd = bis_globaltimer();
                    give_up = *reinterpret_cast<volatile int *>(a.errflag) != 0 || bis_globaltimer() - t_wd > TRSV_WATCHDOG_NS;
                }
                if (__any_sync(0xffffffffu, give_up)) {
                    atomicExch(a.errflag, 1);
                    ok = false;
                    break;
                }
            }
            if (here && ok) {
#pragma unroll
                for (int j = 0; j < PF; ++j)
                    if (cv[j] >= 0)
#pragma unroll
                        for (int w = 0; w < CW; ++w)
                            sum[w] = add_rn(sum[w], mul_rn(av[j], __longlong_as_double((long long)xv[j][w])));
            }
        }
        // a warp that gave up publishes nothing: its rows stay "not ready" and their readers give up too
        if (mine && ok) {
#pragma unroll
            for (int w = 0; w < CW; ++w) {
                if (!(act >> w & 1u)) continue;
                const double r = div_rn(sub_rn(bb[w], sum[w]), dd);
                __stcg(wk + slot * K + c0 + w, r);
                a.X[(int64_t)row * K + c0 + w] = r;
            }
        }
        __syncwarp();
    }
}

template <int K>
int launch_block_trsv(bis_context *c, const BtrsvArgs &a, double *wk) {
    constexpr int R = BtrsvShape<K>::ROWS;
    block_sptrsv_kernel<K><<<(unsigned int)((a.n_slots + R - 1) / R), 256, 0, c->stream>>>(a, wk);
    BIS_LAUNCH_CHECK(c);
    return 0;
}

} // namespace

static int block_trsv_solve(bis_context *c, const bis_matrix *T, int k, double *X, const double *D, const double *B,
                            const double *active, int want_kind) {
    const char *what = want_kind == 1 ? "bis_block_sptrsv" : "bis_block_bsptrsv";
    BIS_REQUIRE(c != nullptr, "null context");
    BIS_REQUIRE(c->nranks == 1, "multi-RHS entry points are single-GPU only (distributed context)");
    BIS_REQUIRE(k >= 1 && k <= BIS_BLOCK_MAX_K, "multi-RHS: k = %d outside [1, %d]", k, BIS_BLOCK_MAX_K);
    BIS_REQUIRE(T && D, "%s: null argument", what);
    BIS_REQUIRE(X && (reinterpret_cast<uintptr_t>(X) & 15) == 0, "multi-RHS: X is null or not 16-byte aligned");
    BIS_REQUIRE(B && (reinterpret_cast<uintptr_t>(B) & 15) == 0, "multi-RHS: B is null or not 16-byte aligned");
    BIS_REQUIRE(T->triangular == want_kind, "%s: matrix is not the %s strictly-triangular factor this call needs", what,
                want_kind == 1 ? "lower" : "upper");
    BIS_REQUIRE(!T->distributed, "%s: triangular sweeps do not shard (single-GPU only)", what);
    BisNvtxRange nvtx_range(want_kind == 1 ? "block-sptrsv" : "block-backwards-sptrsv");
    BIS_CUDA(cudaSetDevice(c->device));
    if (T->n_rows == 0) return 0;
    BIS_CHECK(bis_ensure_levels(c, T));
    LevelSets &lv = T->lv;
    const int64_t need = lv.n_slots * k;
    if (lv.bw_k < k) {   // (re)allocated for the largest k so far; both arrays count as dirty until filled or reset
        BIS_REQUIRE(!c->capturing, "%s: the first solve with %d columns must not be recorded into a graph", what, k);
        BIS_CUDA(cudaStreamSynchronize(c->stream));
        cudaFree(lv.d_bw[0]);
        cudaFree(lv.d_bw[1]);
        lv.d_bw[0] = lv.d_bw[1] = nullptr;
        lv.bw_k = 0;
        BIS_CUDA(bis_cuda_malloc(&lv.d_bw[0], sizeof(double) * (size_t)need));
        BIS_CUDA(bis_cuda_malloc(&lv.d_bw[1], sizeof(double) * (size_t)need));
        lv.bw_k = k;
        lv.bw_dirty[0] = lv.bw_dirty[1] = need;
        lv.bw_epoch = c->graph_epoch;
    }
    const int64_t full = lv.n_slots * lv.bw_k;
    if (lv.bw_epoch != c->graph_epoch || c->capturing) {   // a graph replay may have used either array since
        lv.bw_dirty[0] = lv.bw_dirty[1] = full;
        lv.bw_epoch = c->graph_epoch;
    }
    BtrsvArgs a;
    a.n_slots = lv.n_slots;
    a.slot_row = lv.d_slot_row;
    a.slot_level = lv.d_slot_level;
    a.gate = c->opt_trsv_gates ? reinterpret_cast<const int4 *>(lv.d_slot_gate) : nullptr;
    trsv_wait_params(c, a.gate_sleep, &a.poll_ns);
    a.rp = lv.d_rp;
    a.col = lv.d_col;
    a.val = lv.d_val;
    a.ticket = lv.d_ticket;
    a.errflag = c->d_errflag;
    a.X = X;
    a.D = D;
    a.B = B;
    a.active = active;
    BIS_CHECK(bis_prof_begin(c, BIS_PROF_SPTRSV));
    int p = lv.bw_dirty[0] == 0 ? 0 : (lv.bw_dirty[1] == 0 ? 1 : -1);
    if (p < 0) {   // neither is known to be clean: inside a graph, after one, or on first use
        const int64_t cnt = std::max(lv.bw_dirty[0], need);
        trsv_fill_sentinel_kernel<<<bis_blocks_for(cnt, 1024, c->sm_count * 8), 256, 0, c->stream>>>(cnt, lv.d_bw[0]);
        BIS_LAUNCH_CHECK(c);
        lv.bw_dirty[0] = 0;
        p = 0;
    }
    a.w_clean = lv.d_bw[1 - p];
    // this solve leaves values in [0, need) of its array and resets [0, need) of the other one
    lv.bw_dirty[p] = need;
    lv.bw_dirty[1 - p] = c->capturing ? full : (lv.bw_dirty[1 - p] <= need ? 0 : lv.bw_dirty[1 - p]);
    BIS_CUDA(cudaMemsetAsync(lv.d_ticket, 0, sizeof(unsigned int), c->stream));
    int rc = 2;
    switch (k) {
#define BIS_BTRSV_CASE(KK) case KK: rc = launch_block_trsv<KK>(c, a, lv.d_bw[p]); break;
    BIS_BTRSV_CASE(1) BIS_BTRSV_CASE(2) BIS_BTRSV_CASE(3) BIS_BTRSV_CASE(4) BIS_BTRSV_CASE(5) BIS_BTRSV_CASE(6)
    BIS_BTRSV_CASE(7) BIS_BTRSV_CASE(8) BIS_BTRSV_CASE(9) BIS_BTRSV_CASE(10) BIS_BTRSV_CASE(11) BIS_BTRSV_CASE(12)
    BIS_BTRSV_CASE(13) BIS_BTRSV_CASE(14) BIS_BTRSV_CASE(15) BIS_BTRSV_CASE(16)
#undef BIS_BTRSV_CASE
    }
    BIS_CHECK(rc);
    return bis_prof_end(c, BIS_PROF_SPTRSV);
}

extern "C" int bis_block_sptrsv(bis_context *c, const bis_matrix *L, int k, double *X, const double *D, const double *B,
                                const double *active) {
    return block_trsv_solve(c, L, k, X, D, B, active, 1);
}
extern "C" int bis_block_bsptrsv(bis_context *c, const bis_matrix *U, int k, double *X, const double *D, const double *B,
                                 const double *active) {
    return block_trsv_solve(c, U, k, X, D, B, active, 2);
}

// two_stage_gauss_seidel, kernels.hpp:312-333: a truncated Neumann series for (D + T)^-1 -- SpMV only, no
// dependency chain.  PRECOND_INNER_ITERS is a compile-time -D of the reference (0 in its default build); here
// the context option "precond_inner_iters".  work and tmp trade places locally, as the reference's by-value
// std::swap does; one fused launch per inner iteration (bis_spmv_two_stage).
static int two_stage_gauss_seidel(bis_context *c, const bis_matrix *strict, double *tmp, double *work,
                                  const double *D_inv, const double *in, double *out, int64_t n) {
    BIS_CHECK(bis_elemwise_mult_vectors(c, work, D_inv, in, n, 1.0));
    BIS_CHECK(bis_copy_vector(c, out, work, n));
    const int inner = c->opt_precond_inner_iters;
    if (inner > 0) BIS_REQUIRE(strict && tmp, "bis_apply_preconditioner: 2st with inner iterations needs the strict factor and tmp");
    for (int it = 1; it <= inner; ++it) {
        BIS_CHECK(bis_spmv_two_stage(c, strict, D_inv, work, tmp, out));
        std::swap(work, tmp);
    }
    return 0;
}

// apply_preconditioner, kernels.hpp:336-414 with PRECOND_OUTER_ITERS = 1 (CMakeLists.txt:24); the inner
// iterations of the two-stage variants follow the context option "precond_inner_iters" (reference default 0).
extern "C" int bis_apply_preconditioner(bis_context *c, int precond, int64_t n,
                                        const bis_matrix *L, const bis_matrix *U,
                                        const double *A_D, const double *A_D_inv,
                                        const double *L_D, const double *U_D, double *out,
                                        double *in, double *tmp, double *work) {
    BIS_REQUIRE(c && out && in, "bis_apply_preconditioner: null argument");
    switch (precond) {
    case BIS_PRECOND_JACOBI:
        return bis_elemwise_div_vectors(c, out, in, A_D, n, 1.0);
    case BIS_PRECOND_GS:
        return bis_sptrsv(c, L, out, A_D, in);
    case BIS_PRECOND_BGS:
        return bis_bsptrsv(c, U, out, A_D, in);
    case BIS_PRECOND_SGS:
        BIS_REQUIRE(tmp, "bis_apply_preconditioner: sgs needs tmp");
        // tmp <- D (L+D)^-1 in: the multiply rides in the forward solve's store (same rounding: the
        // reference's elemwise_mult_vectors with scale 1.0 is one rounded product)
        BIS_CHECK(trsv_solve(c, L, tmp, A_D, in, 1, /*post_mul_d=*/1));
        return bis_bsptrsv(c, U, out, A_D, tmp);                    // out <- (D+U)^-1 tmp
    case BIS_PRECOND_2ST:
        BIS_REQUIRE(work && A_D_inv, "bis_apply_preconditioner: 2st needs work and A_D_inv");
        return two_stage_gauss_seidel(c, L, tmp, work, A_D_inv, in, out, n);
    case BIS_PRECOND_S2ST:
        BIS_REQUIRE(work && A_D_inv, "bis_apply_preconditioner: s2st needs work and A_D_inv");
        BIS_CHECK(two_stage_gauss_seidel(c, L, tmp, work, A_D_inv, in, out, n));
        BIS_CHECK(bis_elemwise_mult_vectors(c, out, out, A_D, n, 1.0));
        return two_stage_gauss_seidel(c, U, tmp, work, A_D_inv, out, out, n);
    case BIS_PRECOND_ILU0:
        BIS_REQUIRE(tmp, "bis_apply_preconditioner: ilu0 needs tmp");
        BIS_CHECK(bis_sptrsv(c, L, tmp, L_D, in));   // tmp <- L^-1 in (L_D == 1)
        return bis_bsptrsv(c, U, out, U_D, tmp);     // out <- U^-1 tmp
    case BIS_PRECOND_NONE:
        return bis_copy_vector(c, out, in, n);
    default:
        bis_set_error("bis_apply_preconditioner: unknown preconditioner %d", precond);
        return 2;
    }
}
