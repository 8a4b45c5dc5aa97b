// bis_spmv_win.cuh -- SpMV variant 3: everything a tile needs arrives by TMA,
// x included ("windowed x").
//
// Variant 2 (bis_spmv_tma.cuh) still gathers x[col] from global memory; its ncu
// profile shows the SM waiting on exactly those gathers (long_scoreboard on the
// consuming DMUL) and the L1 data pipe ~80 % busy.  Here the x values a tile of R
// rows touches are described ONCE per matrix as a short list of contiguous column
// windows (a 27-point stencil tile needs 9 windows of R+2 values), and every
// nonzero gets a 16-bit index into the tile's concatenated windows.  A producer
// warp then fetches, per tile, val[], lidx[], the row_ptr slice and the x windows
// with bulk copies (cp.async.bulk -> mbarrier complete_tx); consumer warps wait on
// the "full" barrier, walk one row per thread entirely out of shared memory --
// in-order unfused multiply/add, the reference's summation order, bit-identical to
// native_spmv (kernels.hpp:22-42) -- and release the stage through an "empty"
// barrier.  No thread ever waits on a global load inside the tile loop.
//
// HBM bytes per nonzero drop from 12 (val + col) to 10 (val + lidx); the windows
// are re-read from L2.  The tile format is an acceleration structure derived from
// the CRS arrays, which stay resident and authoritative; matrices whose tiles need
// more than WIN_MAXSEG windows (unstructured sparsity) keep using variant 2.
#pragma once

#include <type_traits>

#include "bis_device.cuh"
#include "bis_spmv_tma.cuh"

constexpr int WIN_MAXSEG = 28;       // x windows per tile (one producer lane each)
constexpr int WIN_GAP = 8;           // columns closer than this share a window
constexpr int WIN_BUILD_THREADS = 256;
constexpr int WIN_FAST_HASH = 128;   // hash slots of the fast path (distinct col - row offsets of a tile)
constexpr int WIN_FAST_OFFS = 64;    // ... and how many distinct offsets it accepts
constexpr int WIN_FAST_EMPTY = (int)0x80000000;

// ---- build: one CTA per tile ---------------------------------------------------------------
struct WinBuildArgs {
    const void *rp;
    const int *col;
    int64_t n_rows;
    int64_t n_owned;      // columns >= n_owned are ghosts (separate base pointer)
    int R;
    int sort_cap;         // power of two >= max nonzeros per tile
    int *seg_start;       // [n_tiles * WIN_MAXSEG]  >= 0: owned column ; < 0: ~ghost index
    unsigned short *seg_len;   // [n_tiles * WIN_MAXSEG] doubles (even)
    unsigned short *seg_off;   // [n_tiles * WIN_MAXSEG] offset into the tile's window buffer
    int *nseg;            // [n_tiles]
    unsigned short *lidx; // [nnz]
    int *status;          // [0] = max window length over tiles, [1] = 1 if some tile is not representable
};

template <typename RP>
__global__ void __launch_bounds__(WIN_BUILD_THREADS) win_build_kernel(WinBuildArgs a) {
    extern __shared__ int s_keys[];                 // [sort_cap]
    __shared__ int s_start[WIN_MAXSEG + 1];         // aligned first column (global numbering) of each window
    __shared__ int s_end[WIN_MAXSEG + 1];           // aligned one-past-last
    __shared__ int s_off[WIN_MAXSEG + 1];
    __shared__ int s_n;
    const RP *__restrict__ rp = static_cast<const RP *>(a.rp);
    const int64_t tile = blockIdx.x;
    const int64_t r0 = tile * a.R;
    int64_t r1 = r0 + a.R;
    if (r1 > a.n_rows) r1 = a.n_rows;
    const int64_t s = (int64_t)rp[r0], e = (int64_t)rp[r1];
    const int m = (int)(e - s);
    const int no = (int)a.n_owned;
    // ---- fast path (banded / stencil tiles without ghost columns): the windows follow from the DISTINCT OFFSETS
    // col - row of the tile.  Offset d contributes the columns [r0 + d, r1 - 1 + d]; offsets closer than the tile is
    // long share a window.  The windows may be supersets of the exact ones (rows at a domain boundary lack some
    // neighbours): harmless, every column a row reads is covered.  More than WIN_FAST_OFFS distinct offsets, a ghost
    // column, or a full hash table: the sort below decides.
    __shared__ int s_hash[WIN_FAST_HASH];
    __shared__ int s_list[WIN_FAST_HASH];
    __shared__ int s_sorted[WIN_FAST_OFFS];
    __shared__ int s_nlist, s_fail, s_fast_runs;
    for (int i = threadIdx.x; i < WIN_FAST_HASH; i += blockDim.x) s_hash[i] = WIN_FAST_EMPTY;
    if (threadIdx.x == 0) {
        s_nlist = 0;
        s_fail = 0;
        s_fast_runs = -1;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
        const int c = a.col[s + i];
        if (c >= no) {
            s_fail = 1;
            continue;
        }
        // the row of nonzero s + i: last row whose rp <= s + i
        int lo = 0, hi = (int)(r1 - r0) - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if ((int64_t)rp[r0 + mid] <= s + i) lo = mid;
            else hi = mid - 1;
        }
        const int d = c - (int)(r0 + lo);
        unsigned int h = ((unsigned int)d * 2654435761u) >> 25;      // 7 bits
        int probes = 0;
        for (;; h = (h + 1) & (WIN_FAST_HASH - 1)) {
            const int v = *reinterpret_cast<volatile int *>(&s_hash[h]);
            if (v == d) break;
            if (v == WIN_FAST_EMPTY) {
                const int old = atomicCAS(&s_hash[h], WIN_FAST_EMPTY, d);
                if (old == WIN_FAST_EMPTY || old == d) break;
            }
            if (++probes >= WIN_FAST_HASH) {
                s_fail = 1;
                break;
            }
        }
    }
    __syncthreads();
    if (!s_fail) {
        for (int i = threadIdx.x; i < WIN_FAST_HASH; i += blockDim.x)
            if (s_hash[i] != WIN_FAST_EMPTY) s_list[atomicAdd(&s_nlist, 1)] = s_hash[i];
    }
    __syncthreads();
    const int n_offs = s_nlist;
    const bool fast = !s_fail && n_offs >= 1 && n_offs <= WIN_FAST_OFFS;
    if (fast) {
        // rank sort of the distinct offsets
        for (int i = threadIdx.x; i < n_offs; i += blockDim.x) {
            const int v = s_list[i];
            int rank = 0;
            for (int j = 0; j < n_offs; ++j) rank += s_list[j] < v ? 1 : 0;
            s_sorted[rank] = v;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            const int span = (int)(r1 - r0) - 1 + WIN_GAP;
            int nrun = 0;
            bool too_many_runs = false;
            int dmin = s_sorted[0], dmax = s_sorted[0];
            for (int i = 1; i <= n_offs; ++i) {
                if (i < n_offs && s_sorted[i] - dmax <= span) {
                    dmax = s_sorted[i];
                    continue;
                }
                if (nrun >= WIN_MAXSEG) {
                    too_many_runs = true;
                    break;
                }
                long long first = (long long)r0 + dmin, last = (long long)r1 - 1 + dmax;
                if (first < 0) first = 0;
                if (last > no - 1) last = no - 1;
                s_start[nrun] = (int)first;
                s_end[nrun] = (int)last;
                ++nrun;
                if (i < n_offs) dmin = dmax = s_sorted[i];
            }
            s_fast_runs = too_many_runs ? -1 : nrun;
        }
    }
    __syncthreads();
    const bool use_fast = s_fast_runs >= 0;
    if (!use_fast) {
    for (int i = threadIdx.x; i < a.sort_cap; i += blockDim.x) s_keys[i] = i < m ? a.col[s + i] : 0x7fffffff;
    __syncthreads();
    // bitonic sort, ascending
    for (int k = 2; k <= a.sort_cap; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < a.sort_cap; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const int x = s_keys[i], y = s_keys[ixj];
                    const bool up = (i & k) == 0;
                    if ((x > y) == up) {
                        s_keys[i] = y;
                        s_keys[ixj] = x;
                    }
                }
            }
            __syncthreads();
        }
    }
    // windows: maximal runs of sorted columns with gaps <= WIN_GAP, never across the owned/ghost border.
    // Parallel: every thread flags the run starts in its slice of the sorted keys, a block scan numbers
    // the runs, the first / last key of each run is written by the thread that sees it.
    __shared__ int s_warp[WIN_BUILD_THREADS / 32];
    __shared__ int s_total;
    const int per = (a.sort_cap + WIN_BUILD_THREADS - 1) / WIN_BUILD_THREADS;
    const int i0 = threadIdx.x * per, i1 = min(i0 + per, m);
    auto is_start = [&](int i) {
        if (i == 0) return true;
        const int p = s_keys[i - 1], c = s_keys[i];
        return (c - p > WIN_GAP) || (p < no && c >= no);
    };
    int cnt = 0;
    for (int i = i0; i < i1; ++i) cnt += is_start(i) ? 1 : 0;
    int incl = cnt;
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if ((int)(threadIdx.x & 31) >= o) incl += v;
    }
    if ((threadIdx.x & 31) == 31) s_warp[threadIdx.x >> 5] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int w = 0; w < WIN_BUILD_THREADS / 32; ++w) {
            const int v = s_warp[w];
            s_warp[w] = run;
            run += v;
        }
        s_total = run;
    }
    __syncthreads();
    const int n_runs = s_total;
    const bool too_many = n_runs > WIN_MAXSEG;
    if (!too_many) {
        int idx = s_warp[threadIdx.x >> 5] + incl - cnt - 1;   // index of the run open at the slice start
        for (int i = i0; i < i1; ++i) {
            if (is_start(i)) {
                ++idx;
                s_start[idx] = s_keys[i];                       // first key of the run (aligned below)
            }
            if (i == m - 1 || is_start(i + 1)) s_end[idx] = s_keys[i];   // last key of the run
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) s_fast_runs = too_many ? -2 : n_runs;
    }   // sort path
    __syncthreads();
    // each window is widened to even bounds relative to its base pointer (16-byte bulk copies)
    if (threadIdx.x == 0) {
        int off = 0;
        bool bad = s_fast_runs < 0;
        const int n = bad ? 0 : s_fast_runs;
        for (int q = 0; q < n; ++q) {
            const int first = s_start[q], last = s_end[q];
            const int base = first >= no ? no : 0;
            const int lo = base + ((first - base) & ~1);
            const int hi = base + ((last - base + 2) & ~1);      // one past, even
            s_start[q] = lo;
            s_end[q] = hi;
            s_off[q] = off;
            off += hi - lo;
        }
        if (off > 65534) bad = true;
        s_n = bad ? -1 : n;
        if (bad) atomicExch(a.status + 1, 1);
        else atomicMax(a.status, off);
        a.nseg[tile] = bad ? 0 : n;
    }
    __syncthreads();
    if (threadIdx.x < WIN_MAXSEG) {
        const int q = threadIdx.x;
        const bool live = s_n >= 0 && q < s_n;
        const int lo = live ? s_start[q] : 0;
        a.seg_start[tile * WIN_MAXSEG + q] = !live ? 0 : (lo >= no ? ~(lo - no) : lo);
        a.seg_len[tile * WIN_MAXSEG + q] = (unsigned short)(live ? s_end[q] - lo : 0);
        a.seg_off[tile * WIN_MAXSEG + q] = (unsigned short)(live ? s_off[q] : 0);
    }
    __syncthreads();
    const int n = s_n;
    if (n < 0) return;
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
        const int c = a.col[s + i];
        int lo = 0, hi = n - 1;            // last window whose start <= c
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (s_start[mid] <= c) lo = mid;
            else hi = mid - 1;
        }
        a.lidx[s + i] = (unsigned short)(s_off[lo] + (c - s_start[lo]));
    }
}

// ---- tile order ----------------------------------------------------------------------------------
// The tiles of a launch are processed in the order of a table built once per matrix (bis_spmv.cu:
// win_build_order): per local virtual slab first the tiles that only read columns of their own slab
// (y-blocked through z when the grid is known and a plane of x no longer survives in L2 between its
// uses), then the slab's low and high boundary strips.  The order depends on the GLOBAL problem only,
// and CTA b of the logical grid G takes positions b, b + G, ... of every slab, so the per-(slab, CTA)
// partial sums of a fused dot product are the same numbers at every rank count (bis_internal.cuh).
// Bit 31 of an entry: the tile reads ghost values (the halo exchange must have landed).
constexpr int WIN_ORDER_GHOST = (int)0x80000000u;

struct WinOrderArgs {
    const int *order;            // [n_tiles]
    int n_slab;
    int pos0[BIS_NSLAB + 1];     // positions [pos0[i], pos0[i+1]) belong to local slab i
    int G;                       // logical grid (interleave stride)
    int part_stride;             // partial of (slab i, CTA b) sits at i * part_stride + b
};

// ---- SpMV ----------------------------------------------------------------------------------------
// Distributed SpMV as ONE kernel (peer-memory transport, bis_dist.cu): every CTA first packs its share
// of the boundary values of x and stores them straight into the neighbours' ghost buffers (the CTA
// that finishes last publishes the exchange's epoch in their banks), then the grid sweeps the tiles in
// table order (interiors first), and a CTA's producer warp looks at the senders' flags only when it
// reaches its first tile that reads ghosts -- by then the values have long arrived.  The fused dot
// product and its sum over ranks (block_reduce_finish) close the same kernel.
struct NoHaloFuse {};

struct SpmvWinIn {
    const void *rp;
    const double *val;
    const unsigned short *lidx;
    const int *seg_start;
    const unsigned short *seg_len;
    const unsigned short *seg_off;
    const int *nseg;
    const double *x;
    const double *ghost;
    int64_t n_rows;
    WinOrderArgs ord;
    // value dictionary (WinFormat): when vidx != nullptr a stage receives the 1-byte indices vidx[s..e) instead of
    // val[s..e) and the row walk reads vdict[index] (a copy of the <= 256 entry table in shared memory)
    const unsigned char *vidx;
    const double *vdict;
    int n_dict;
    int val_region;               // bytes of a stage's value part: cap * 8, or cap with the dictionary
    int amask;                    // copies start at element (rp[r0] & ~amask): 7, or 15 with the dictionary (16-byte units)
    int R;                        // rows per tile == consumer threads
    int cap;                      // nonzeros per stage (multiple of 16)
    int xcap;                     // window doubles per stage (even)
    int nstage;                   // stages of the pipeline (tile s lands in stage s % nstage)
    int ngroups;                  // consumer groups (tile s is computed by group s % ngroups); nstage is a multiple of it
    int stage_bytes;
#ifdef BIS_PERF_DEBUG
    int debug;                    // perf experiments only: 1 = consumers skip the row walk, 2 = no x-window copies (results
                                  // invalid); 4 = per-role cycle counters into `stamps` (results valid, see WinStamp)
    unsigned long long *stamps;   // [WIN_NSTAMP], summed over the CTAs
#endif
};
#ifdef BIS_PERF_DEBUG
#define BIS_WIN_DEBUG(in, bit) ((in).debug & (bit))
#else
#define BIS_WIN_DEBUG(in, bit) 0
#endif

// Per-role cycle counters of the -DBIS_PERF_DEBUG build (spmv_debug bit 4; tools/run_spmv_stamps.py).  Producer: lane 0
// of the producer warp; consumers: lane 0 of every consumer warp (a warp's lanes run the same steps).  SM cycles
// (clock64): the phases of a tile are a few hundred cycles, below what the global timer resolves.
enum WinStamp {
    WS_P_EMPTY = 0,     // producer: waiting on a stage's `empty` barrier
    WS_P_ISSUE,         // producer: proxy fence, expect_tx and the bulk-copy instructions of a tile
    WS_P_TILES,         // producer: tiles issued
    WS_P_TOTAL,         // producer: whole tile loop
    WS_C_ORDER,         // consumers: waiting on the next tile id (order table load)
    WS_C_FULL,          // consumers: waiting on a stage's `full` barrier
    WS_C_EPILOAD,       // consumers: waiting on the epilogue operand load issued before the `full` wait
    WS_C_WALK,          // consumers: row walk and epilogue stores
    WS_C_TILES,         // consumers: tiles, summed over warps
    WS_C_TOTAL,         // consumers: whole tile loop, summed over warps
    WIN_NSTAMP = 16     // the host writes the launch's grid size into the last slot
};

// stage layout: [val cap*8 | vidx cap][xwin xcap*8][rp (R+4)*8][lidx cap*2], every part 16-byte aligned
constexpr int WIN_MAX_THREADS = 544;   // consumer groups (R x nstage <= 512) + the producer warp

// This CTA's sequence of tiles: the s-th one is position pos0[i] + b + (s - cum[i]) * G of slab i.
struct WinSeq {
    int cum[BIS_NSLAB + 1];
    __device__ __forceinline__ void init(const WinOrderArgs &o, int b) {
        cum[0] = 0;
#pragma unroll
        for (int i = 0; i < BIS_NSLAB; ++i) {
            int c = 0;
            if (i < o.n_slab) {
                const int len = o.pos0[i + 1] - o.pos0[i];
                c = len > b ? (len - b + o.G - 1) / o.G : 0;
            }
            cum[i + 1] = cum[i] + c;
        }
    }
    __device__ __forceinline__ int total() const { return cum[BIS_NSLAB]; }
    __device__ __forceinline__ int slab_of(int s) const {
        int i = 0;
#pragma unroll
        for (int k = 1; k < BIS_NSLAB; ++k) i += (s >= cum[k]) ? 1 : 0;
        return i;
    }
    __device__ __forceinline__ int pos(const WinOrderArgs &o, int b, int s) const {
        const int i = slab_of(s);
        return o.pos0[i] + b + (s - cum[i]) * o.G;
    }
};

template <typename RP, class Epi, bool DIST = false>
__global__ void __launch_bounds__(WIN_MAX_THREADS, 1)
spmv_win_kernel(SpmvWinIn in, Epi epi, RedArgs ra, typename std::conditional<DIST, HaloFuse, NoHaloFuse>::type hf) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw);            // [MAX_STAGES]
    uint64_t *empty = full + tma::MAX_STAGES;                           // [MAX_STAGES]
    unsigned char *stages = smem_raw + 128;
    const int R = in.R;
    // one consumer GROUP (R threads) per stage: group g computes the tiles that land in stage g, so
    // while one group walks its rows the next tile's group is already waiting on its own barrier and
    // starts the moment its copies land -- nstage tiles can be in the compute phase at once
    const int n_cons_warps = R >> 5;                  // per group
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool producer = warp == n_cons_warps * in.ngroups;       // the last warp
    const int group = warp / n_cons_warps;
    const int tid_g = (int)threadIdx.x - group * R;   // thread index inside its group
    WinSeq seq;
    seq.init(in.ord, (int)blockIdx.x);
    const int my_tiles = seq.total();

    double acc[Epi::NRED > 0 ? Epi::NRED : 1];
#pragma unroll
    for (int q = 0; q < (Epi::NRED > 0 ? Epi::NRED : 1); ++q) acc[q] = 0.0;

    __shared__ double s_dict[256];
    if (in.vidx)
        for (int i = threadIdx.x; i < in.n_dict; i += blockDim.x) s_dict[i] = in.vdict[i];
    if (threadIdx.x == 0) {
        for (int s = 0; s < in.nstage; ++s) {
            tma::mbar_init(&full[s], 1);
            tma::mbar_init(&empty[s], n_cons_warps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if constexpr (DIST) {
        // pack + publish (the protocol of pack_peer_kernel, bis_dist.cu)
        __shared__ bool s_last;
        const int t = threadIdx.x;
        if (blockIdx.x == 0 && t < hf.n_ranks && t != hf.me)
            *reinterpret_cast<volatile unsigned long long *>(hf.ack_out[t]) = hf.epoch;
        if (t < hf.n_dst && hf.epoch >= 2) {
            const volatile unsigned long long *ack = hf.ack_in + hf.dst_rank[t];
            const unsigned long long t0 = bis_globaltimer();
            while (*ack + 1 < hf.epoch) {
                if (bis_globaltimer() - t0 > BIS_PEER_TIMEOUT_NS) {
                    atomicExch(hf.errflag, 30 + hf.dst_rank[t]);
                    break;
                }
            }
        }
        __syncthreads();
        const int64_t n_send = hf.seg_off[hf.n_dst];
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + t; i < n_send; i += (int64_t)gridDim.x * blockDim.x) {
            int d = 0;
            while (i >= hf.seg_off[d + 1]) ++d;
            hf.dst[d][i - hf.seg_off[d]] = in.x[hf.send_idx[i]];
        }
        __threadfence_system();
        __syncthreads();
        if (t == 0) s_last = (atomicAdd(hf.ticket, 1u) == gridDim.x - 1);
        __syncthreads();
        if (s_last) {
            if (t < hf.n_dst) {
                __threadfence_system();
                *reinterpret_cast<volatile unsigned long long *>(hf.dst_flag[t]) = hf.epoch;
            }
            if (t == 0) *hf.ticket = 0u;
        }
    }

    if (producer) {
        const RP *__restrict__ rp = static_cast<const RP *>(in.rp);
        const uint64_t pol_stream = tma::policy_evict_first();
        uint64_t pol_keep;
        asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_keep));
        // What this lane copies for one tile: lane 0 val, lane 1 lidx, lane 2 the row_ptr slice,
        // lanes 3.. one x window each.  Everything the copies are described by comes from global
        // memory -- the tile id from the order table, then row_ptr and the window table -- so the
        // tile ids are requested 2*PDEPTH and the descriptors PDEPTH tiles ahead: the producer never
        // sits on a global-load latency between two tiles.
        // Raw words are only LOADED ahead of time; nothing is computed from them until the next
        // pipeline step (a dependent instruction right after a load would stall the warp for a full
        // memory latency per tile and serialise the whole pipeline).
        struct Desc {
            RP a, b;                 // rp[r0], rp[r1]            (lanes 0, 1)
            int start;               // window start              (lanes 3..)
            unsigned short len, off; // window length / offset    (lanes 3..)
            int tile;                // raw order entry
        };
        const uint32_t off_xw = (uint32_t)in.val_region;
        const uint32_t off_rp = off_xw + (uint32_t)in.xcap * 8u;
        const uint32_t off_li = off_rp + (uint32_t)(R + 4) * 8u;
        auto tile_rows = [&](int tile, int64_t &r0, int64_t &r1) {
            r0 = (int64_t)tile * R;
            r1 = r0 + R;
            if (r1 > in.n_rows) r1 = in.n_rows;
        };
        auto load_order = [&](int s) -> int {
            return s < my_tiles ? in.ord.order[seq.pos(in.ord, (int)blockIdx.x, s)] : 0;
        };
        // loads only -- no conversion, no arithmetic on the loaded words (see above)
        auto load_desc = [&](int s, int raw, Desc &d) {
            d.a = 0;
            d.b = 0;
            d.start = 0;
            d.len = 0;
            d.off = 0;
            d.tile = raw;
            if (s >= my_tiles) return;
            const int tile = raw & ~WIN_ORDER_GHOST;
            int64_t r0, r1;
            tile_rows(tile, r0, r1);
            if (lane < 2) {
                d.a = rp[r0];
                d.b = rp[r1];
            } else if (lane >= 3 && lane - 3 < WIN_MAXSEG) {
                const int64_t q = (int64_t)tile * WIN_MAXSEG + (lane - 3);
                d.start = in.seg_start[q];
                d.len = in.seg_len[q];
                d.off = in.seg_off[q];
            }
        };
        [[maybe_unused]] bool halo_seen = false;
#ifdef BIS_PERF_DEBUG
        long long pst[4] = {0, 0, 0, 0};
        const long long t_p0 = clock64();
#endif
        auto issue = [&](int s, const Desc &d) {
            if constexpr (DIST) {
                // first tile of this CTA that reads ghosts: the senders' values must have landed
                if (!halo_seen && (d.tile & WIN_ORDER_GHOST)) {
                    const unsigned long long t_wait0 = bis_globaltimer();
                    for (int q = 0; q < hf.n_src; ++q) {
                        const volatile unsigned long long *f = hf.flag_in + hf.src_rank[q];
                        const unsigned long long t0 = bis_globaltimer();
                        while (*f < hf.epoch) {
                            if (bis_globaltimer() - t0 > BIS_PEER_TIMEOUT_NS) {
                                atomicExch(hf.errflag, 40 + hf.src_rank[q]);
                                break;
                            }
                        }
                    }
                    __threadfence_system();
                    // the bulk copies below read the ghosts through the async proxy
                    asm volatile("fence.proxy.async.global;" ::: "memory");
                    halo_seen = true;
                    if (blockIdx.x == 0 && lane == 0 && hf.waitstat) {
                        hf.waitstat[2] += bis_globaltimer() - t_wait0;
                        hf.waitstat[3] += 1ull;
                    }
                }
            }
            const int st = s % in.nstage;
            int64_t r0, r1;
            tile_rows(d.tile & ~WIN_ORDER_GHOST, r0, r1);
            const void *src = nullptr;
            uint32_t bytes = 0, dst = 0;
            if (lane < 2) {
                const int64_t am = in.amask;
                const int64_t s_al = (int64_t)d.a & ~am;
                const uint32_t n_el = (uint32_t)((((int64_t)d.b + am) & ~am) - s_al);
                if (lane == 0) {
                    if (in.vidx) {
                        src = in.vidx + s_al;
                        bytes = n_el;
                    } else {
                        src = in.val + s_al;
                        bytes = n_el * 8u;
                    }
                } else {
                    src = in.lidx + s_al;
                    bytes = n_el * 2u;
                    dst = off_li;
                }
            } else if (lane == 2) {
                src = rp + r0;
                bytes = (uint32_t)(((r1 - r0 + 1) + 3) & ~(int64_t)3) * (uint32_t)sizeof(RP);
                dst = off_rp;
            } else if (d.len && !BIS_WIN_DEBUG(in, 2)) {
                src = d.start >= 0 ? in.x + d.start : in.ghost + (~d.start);
                bytes = (uint32_t)d.len * 8u;
                dst = off_xw + (uint32_t)d.off * 8u;
            }
            uint32_t total = bytes;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
#ifdef BIS_PERF_DEBUG
            const long long t_w0 = clock64();
#endif
            // the stage must have been released by every consumer warp
            if (s >= in.nstage) tma::mbar_wait(&empty[st], (uint32_t)(((s / in.nstage) - 1) & 1));
#ifdef BIS_PERF_DEBUG
            const long long t_w1 = clock64();
#endif
            if (s >= in.nstage) tma::fence_reads_before_bulk_write();
            unsigned char *sb = stages + (size_t)st * in.stage_bytes;
            if (lane == 0) tma::mbar_expect_tx(&full[st], total);
            __syncwarp();
            if (bytes) tma::bulk_g2s(sb + dst, src, bytes, &full[st], lane < 3 ? pol_stream : pol_keep);
#ifdef BIS_PERF_DEBUG
            __syncwarp();
            pst[WS_P_EMPTY] += t_w1 - t_w0;
            pst[WS_P_ISSUE] += clock64() - t_w1;
            pst[WS_P_TILES] += 1;
#endif
        };
        constexpr int PDEPTH = 4;
        int tq[2 * PDEPTH];     // order entries of tiles s .. s + 7
        Desc dq[PDEPTH];        // descriptors of tiles s .. s + 3
#pragma unroll
        for (int u = 0; u < 2 * PDEPTH; ++u) tq[u] = load_order(u);
#pragma unroll
        for (int u = 0; u < PDEPTH; ++u) load_desc(u, tq[u], dq[u]);
        for (int s0 = 0; s0 < my_tiles; s0 += 2 * PDEPTH) {
#pragma unroll
            for (int u = 0; u < 2 * PDEPTH; ++u) {
                const int s = s0 + u;
                if (s < my_tiles) issue(s, dq[u % PDEPTH]);
                // slot u of tq held tile s: refill it with tile s + 8; the descriptor slot takes tile s + 4,
                // whose id was requested at least four tiles ago
                load_desc(s + PDEPTH, tq[(u + PDEPTH) % (2 * PDEPTH)], dq[u % PDEPTH]);
                tq[u] = load_order(s + 2 * PDEPTH);
            }
        }
#ifdef BIS_PERF_DEBUG
        if (in.stamps && lane == 0) {
            pst[WS_P_TOTAL] = clock64() - t_p0;
            for (int q = 0; q < 4; ++q) atomicAdd(in.stamps + q, (unsigned long long)pst[q]);
        }
#endif
    } else {
        [[maybe_unused]] int cur_slab = 0;
        // the slab-end partial of a fused reduction is formed by the consumer warps alone (the producer
        // is still copying): consumer-only named barrier, warp sums parked by LOGICAL warp (the group that
        // took the slab's first tile counts as group 0, so the sum is independent of where in this CTA's
        // sequence the slab starts), two parities so that one barrier per slab suffices
        __shared__ double s_wsum[2][Epi::NRED > 0 ? Epi::NRED : 1][32];
        const int n_cons_threads = R * in.ngroups;
        auto close_slab = [&](int slab) {
            if constexpr (Epi::NRED > 0) {
                const int par = slab & 1;
                const int g0 = seq.cum[slab] % in.ngroups;                    // group that got the slab's first tile
                const int lgroup = (group - g0 + in.ngroups) % in.ngroups;
                const int lwarp = lgroup * n_cons_warps + (warp - group * n_cons_warps);
#pragma unroll
                for (int q = 0; q < Epi::NRED; ++q) {
                    const double v = warp_sum(acc[q]);
                    if (lane == 0) s_wsum[par][q][lwarp] = v;
                    acc[q] = 0.0;
                }
                asm volatile("bar.sync 1, %0;" ::"r"(n_cons_threads) : "memory");
                if (warp == 0) {
                    const int nw = n_cons_warps * in.ngroups;
#pragma unroll
                    for (int q = 0; q < Epi::NRED; ++q) {
                        double v = lane < nw ? s_wsum[par][q][lane] : 0.0;
                        v = warp_sum(v);
                        if (lane == 0)
                            ra.partials[q * BIS_MAX_RED_BLOCKS + ra.block_offset + slab * in.ord.part_stride + (int)blockIdx.x] = v;
                    }
                }
            }
        };
        int raw_next = group < my_tiles ? in.ord.order[seq.pos(in.ord, (int)blockIdx.x, group)] : 0;
#ifdef BIS_PERF_DEBUG
        long long cst[6] = {0, 0, 0, 0, 0, 0};     // WS_C_ORDER .. WS_C_TOTAL
        const long long t_c0 = clock64();
#endif
        for (int s = group; s < my_tiles; s += in.ngroups) {
            const int st = s % in.nstage;
#ifdef BIS_PERF_DEBUG
            long long t_a = clock64();
            if (in.stamps) {     // consume the tile id now, so that its wait is counted here
                int v;
                asm volatile("add.s32 %0, %1, 1;" : "=r"(v) : "r"(raw_next));
                asm volatile("" ::"r"(v));
                const long long t_b = clock64();
                cst[0] += t_b - t_a;
                t_a = t_b;
            }
#endif
            const int tile = raw_next & ~WIN_ORDER_GHOST;
            if constexpr (Epi::NRED > 0) {
                const int slab = seq.slab_of(s);
                while (cur_slab < slab) close_slab(cur_slab++);
            }
            // the next tile's id is requested a whole tile ahead
            if (s + in.ngroups < my_tiles) raw_next = in.ord.order[seq.pos(in.ord, (int)blockIdx.x, s + in.ngroups)];
            const int64_t row = (int64_t)tile * R + tid_g;
            const unsigned char *sb = stages + (size_t)st * in.stage_bytes;
            const double *__restrict__ sval = reinterpret_cast<const double *>(sb);
            const unsigned char *__restrict__ svi = sb;
            const double *__restrict__ sxw = reinterpret_cast<const double *>(sb + in.val_region);
            const RP *__restrict__ srp = reinterpret_cast<const RP *>(sxw + in.xcap);
            const unsigned short *__restrict__ sli =
                reinterpret_cast<const unsigned short *>(reinterpret_cast<const unsigned char *>(srp) + (size_t)(R + 4) * 8);
            EpiPre pre{0.0, 0.0, 0.0};
            if (row < in.n_rows) pre = epi.load(row);   // in flight during the wait and the row walk
#ifdef BIS_PERF_DEBUG
            const long long t_f0 = clock64();
#endif
            tma::mbar_wait(&full[st], (uint32_t)((s / in.nstage) & 1));
#ifdef BIS_PERF_DEBUG
            long long t_f1 = clock64();
            if (in.stamps) {
                cst[1] += t_f1 - t_f0;
                double v;
                asm volatile("add.f64 %0, %1, %2;" : "=d"(v) : "d"(pre.a), "d"(pre.b));
                asm volatile("add.f64 %0, %0, %1;" : "+d"(v) : "d"(pre.c));
                asm volatile("" ::"d"(v));
                const long long t_f2 = clock64();
                cst[2] += t_f2 - t_f1;
                t_f1 = t_f2;
            }
            (void)t_a;
#endif
            if (row < in.n_rows && !BIS_WIN_DEBUG(in, 1)) {
                const int64_t base = (int64_t)srp[0] & ~(int64_t)in.amask;
                const int ks = (int)((int64_t)srp[tid_g] - base);
                const int ke = (int)((int64_t)srp[tid_g + 1] - base);
                double sum = 0.0;
                int k = ks;
                if (in.vidx) {          // the same walk with the value looked up by its 1-byte index (warp-uniform)
                    for (; k + 9 <= ke; k += 9) {
                        double a[9], xv[9];
#pragma unroll
                        for (int u = 0; u < 9; ++u) {
                            a[u] = s_dict[svi[k + u]];
                            xv[u] = sxw[sli[k + u]];
                        }
#pragma unroll
                        for (int u = 0; u < 9; ++u) sum = add_rn(sum, mul_rn(a[u], xv[u]));
                    }
                    for (; k < ke; ++k) sum = add_rn(sum, mul_rn(s_dict[svi[k]], sxw[sli[k]]));
                }
                for (; k + 9 <= ke; k += 9) {
                    double a[9], xv[9];
#pragma unroll
                    for (int u = 0; u < 9; ++u) {
                        a[u] = sval[k + u];
                        xv[u] = sxw[sli[k + u]];
                    }
#pragma unroll
                    for (int u = 0; u < 9; ++u) sum = add_rn(sum, mul_rn(a[u], xv[u]));
                }
                for (; k < ke; ++k) sum = add_rn(sum, mul_rn(sval[k], sxw[sli[k]]));
                epi(row, sum, pre, acc);
            }
            __syncwarp();
#ifdef BIS_PERF_DEBUG
            cst[3] += clock64() - t_f1;
            cst[4] += 1;
#endif
            if (lane == 0) tma::mbar_arrive(&empty[st]);
        }
#ifdef BIS_PERF_DEBUG
        if (in.stamps && lane == 0) {
            cst[5] = clock64() - t_c0;
            for (int q = 0; q < 6; ++q) atomicAdd(in.stamps + WS_C_ORDER + q, (unsigned long long)cst[q]);
        }
#endif
        if constexpr (Epi::NRED > 0) {
            while (cur_slab < in.ord.n_slab) close_slab(cur_slab++);
        }
    }
    if constexpr (Epi::NRED > 0) grid_reduce_finish<Epi::NRED>(ra);
}
