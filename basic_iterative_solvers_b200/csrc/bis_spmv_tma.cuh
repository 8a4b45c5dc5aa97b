// bis_spmv_tma.cuh -- SpMV variant 2: TMA-staged, one thread per row.
//
// The nonzeros of a block of consecutive rows are contiguous in CRS, so a tile
// of R rows is fetched by TWO 1-D bulk copies (cp.async.bulk, the TMA engine:
// SASS UBLKCP) -- val[s..e) and col[s..e) -- into shared memory, completion
// signalled on an mbarrier.  HBM is therefore read in large, perfectly
// sequential, fully used bursts that no thread has to wait on instruction by
// instruction; NSTAGE tiles are in flight per CTA.  A tile is then consumed in
// two phases.  (1) All threads form the products p_k = val_k * x[col_k] of the
// whole tile, nonzero-major (conflict-free shared memory, every gather
// independent of every other: the x loads of a tile are all in flight at once),
// and store p_k over val_k.  (2) One thread per row adds ITS products strictly
// left to right.  Separately rounded products added in storage order is exactly
// what the compiled reference does (kernels.hpp:31-36 under GCC's in-order
// `omp simd` reduction), so y is bit-identical to native_spmv; the only
// sequential part left is a chain of <= max_row shared-memory adds.
//
// Grid: persistent, one CTA per SM (x occupancy), each CTA owns a CONTIGUOUS
// run of tiles (static assignment => fused dot products are bit-reproducible,
// and neighbouring tiles reuse x lines in L1).
//
// Shared memory per stage: cap * 12 bytes, cap = R * max_row + 8 (the copies
// start and end on 16-byte boundaries; the arrays are allocated with 4 spare
// elements for that).
#pragma once

#include "bis_device.cuh"

#include <cuda.h>

namespace tma {

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// Before a bulk copy OVERWRITES shared memory that was read with ordinary loads: those reads went through the generic
// proxy, the copy writes through the async proxy, and only this fence orders the two (after whatever barrier told the
// issuing thread that the readers are done).  Seen to matter in bis_sptrsv_wave.cuh.
__device__ __forceinline__ void fence_reads_before_bulk_write() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// 1-D bulk copy global -> shared, bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar,
                                         uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
        "[%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}

// 3-D tensor copy global -> shared of the box at (c0, c1, c2) of `map` (cuTensorMapEncodeTiled); dst 128-byte aligned.
// Elements outside the tensor arrive as zeros and count towards the transaction bytes like the others.
__device__ __forceinline__ void tensor3d_g2s(void *dst, const CUtensorMap *map, int c0, int c1, int c2, uint64_t *bar,
                                             uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint "
        "[%0], [%1, {%2, %3, %4}], [%5], %6;" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}

constexpr int MAX_STAGES = 8;

struct Plan {
    int threads;          // threads per CTA (a multiple of rows)
    int rows;             // rows per tile
    int cap;              // elements per stage
    int nstage;
    int grid;
    int64_t tiles_per_cta;
    size_t smem_bytes;
};

}  // namespace tma

struct SpmvTmaIn {
    const void *rp;
    const int *col;
    const double *val;
    const double *x;
    const double *ghost;
    int64_t n_owned;
    int64_t lo, cnt;          // contiguous row range of this launch
    int64_t tiles_per_cta;
    int cap;
    int nstage;
    int interleave;           // 1: tile j of CTA b is b + j*grid ; 0: b*tiles_per_cta + j
    int rows;                 // rows per tile (blockDim.x is a multiple of it)
};

constexpr int PBATCH = 7;   // independent gathers in flight per thread in phase 1

template <typename RP, bool GHOST, class Epi>
__global__ void __launch_bounds__(1024) spmv_tma_kernel(SpmvTmaIn in, Epi epi, RedArgs ra) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw);                       // [MAX_STAGES]
    double *sval = reinterpret_cast<double *>(smem_raw + 128);                     // [nstage][cap]
    int *scol = reinterpret_cast<int *>(smem_raw + 128 + (size_t)in.nstage * in.cap * sizeof(double));

    const RP *__restrict__ rp = static_cast<const RP *>(in.rp);
    const double *__restrict__ x = in.x;
    const int R = in.rows;            // rows per tile; phase 1 uses all blockDim.x threads
    const int T = blockDim.x;
    const int64_t n_tiles = (in.cnt + R - 1) / R;
    // static tile -> CTA map (bit-reproducible fused reductions).  Interleaved: all CTAs sweep
    // the matrix together, so the x window they gather from is shared in L2; blocked: each CTA
    // owns a contiguous run (x lines are reused in its L1, but the CTAs' windows are disjoint).
    int64_t t_first, t_stride, my_tiles;
    if (in.interleave) {
        t_first = blockIdx.x;
        t_stride = gridDim.x;
        my_tiles = n_tiles > t_first ? (n_tiles - t_first + t_stride - 1) / t_stride : 0;
    } else {
        t_first = (int64_t)blockIdx.x * in.tiles_per_cta;
        t_stride = 1;
        int64_t t_end = t_first + in.tiles_per_cta;
        if (t_end > n_tiles) t_end = n_tiles;
        my_tiles = t_end > t_first ? t_end - t_first : 0;
    }
    const int64_t row_end = in.lo + in.cnt;

    double acc[Epi::NRED > 0 ? Epi::NRED : 1];
#pragma unroll
    for (int q = 0; q < (Epi::NRED > 0 ? Epi::NRED : 1); ++q) acc[q] = 0.0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < in.nstage; ++s) tma::mbar_init(&bars[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    uint64_t policy = 0;
    if (threadIdx.x == 0) policy = tma::policy_evict_first();

    // nonzero range [s, e) of CTA-local tile j (same value in every thread: broadcast loads)
    auto tile_range = [&](int64_t j, int64_t &s, int64_t &e) {
        if (j >= my_tiles) {
            s = e = 0;
            return;
        }
        const int64_t r0 = in.lo + (t_first + j * t_stride) * R;
        int64_t r1 = r0 + R;
        if (r1 > row_end) r1 = row_end;
        s = (int64_t)rp[r0];
        e = (int64_t)rp[r1];
    };
    // producer (thread 0): two bulk copies of tile j's val / col into its stage
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

    // this thread's row of tile j: nonzero range [ks, ke), or row = -1
    auto row_bounds = [&](int64_t j, int64_t &ks, int64_t &ke, int64_t &row) {
        row = in.lo + (t_first + j * t_stride) * R + threadIdx.x;
        if (j < my_tiles && row < row_end && (int)threadIdx.x < R) {
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
        // everything the NEXT tiles need from row_ptr is requested before the wait
        int64_t nts, nte, nks, nke, nrow, is = 0, ie = 0;
        tile_range(j + 1, nts, nte);
        row_bounds(j + 1, nks, nke, nrow);
        if (threadIdx.x == 0) tile_range(j + in.nstage, is, ie);
        EpiPre pre{0.0, 0.0, 0.0};
        if (row >= 0) pre = epi.load(row);   // in flight during the wait and both phases
        tma::mbar_wait(&bars[st], parity);

        const int64_t base = ts & ~(int64_t)3;
        double *__restrict__ sv = sval + (size_t)st * in.cap;
        const int *__restrict__ sc = scol + (size_t)st * in.cap;
        // phase 1: every product p_k = val_k * x[col_k] of the tile, all threads, independent
        // gathers (memory-level parallelism), stored over val_k
        const int k_lo = (int)(ts - base), k_hi = (int)(te - base);
        for (int k0 = k_lo + (int)threadIdx.x; k0 < k_hi; k0 += PBATCH * T) {
            int c[PBATCH];
            double v[PBATCH], xv[PBATCH];
#pragma unroll
            for (int u = 0; u < PBATCH; ++u) {
                const int k = k0 + u * T;
                const bool ok = k < k_hi;
                c[u] = ok ? sc[k] : -1;
                v[u] = ok ? sv[k] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < PBATCH; ++u) {
                if (c[u] < 0) xv[u] = 0.0;
                else if (GHOST && c[u] >= in.n_owned) xv[u] = __ldg(in.ghost + (c[u] - in.n_owned));
                else xv[u] = __ldg(x + c[u]);
            }
#pragma unroll
            for (int u = 0; u < PBATCH; ++u) {
                const int k = k0 + u * T;
                if (k < k_hi) sv[k] = mul_rn(v[u], xv[u]);
            }
        }
        __syncthreads();
        // phase 2: one thread per row adds its products left to right (the reference's order)
        if (row >= 0) {
            double sum = 0.0;
            const int a = (int)(ks - base), b = (int)(ke - base);
            int k = a;
            for (; k + 9 <= b; k += 9) {
                double p[9];
#pragma unroll
                for (int u = 0; u < 9; ++u) p[u] = sv[k + u];
#pragma unroll
                for (int u = 0; u < 9; ++u) sum = add_rn(sum, p[u]);
            }
            for (; k < b; ++k) sum = add_rn(sum, sv[k]);
            epi(row, sum, pre, acc);
        }
        __syncthreads();   // every thread is done with stage `st`
        if (threadIdx.x == 0 && j + in.nstage < my_tiles) {
            // the stage was written through the generic proxy (phase 1): order those writes
            // before the bulk copy (async proxy) overwrites it
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            issue(j + in.nstage, is, ie);
        }
        ts = nts; te = nte; ks = nks; ke = nke; row = nrow;
    }
    if constexpr (Epi::NRED > 0) block_reduce_finish<Epi::NRED>(acc, ra);
}
