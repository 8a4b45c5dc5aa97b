// bis_internal.cuh -- shared declarations of the sm_100a implementation behind
// include/bis_b200.h.  Nothing here is part of the ABI.
#pragma once

#include "bis_b200.h"

#include <cuda_runtime.h>
#include <nccl.h>
#include <nvtx3/nvToolsExt.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

// ---- error plumbing -------------------------------------------------------
void bis_set_error(const char *fmt, ...);

#define BIS_CUDA(call)                                                         \
    do {                                                                       \
        cudaError_t _e = (call);                                               \
        if (_e != cudaSuccess) {                                               \
            bis_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call,   \
                          cudaGetErrorString(_e));                             \
            return 1;                                                          \
        }                                                                      \
    } while (0)

#define BIS_NCCL(call)                                                         \
    do {                                                                       \
        ncclResult_t _r = (call);                                              \
        if (_r != ncclSuccess) {                                               \
            bis_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call,   \
                          ncclGetErrorString(_r));                             \
            return 1;                                                          \
        }                                                                      \
    } while (0)

#define BIS_CHECK(expr)                                                        \
    do {                                                                       \
        int _rc = (expr);                                                      \
        if (_rc != 0)                                                          \
            return _rc;                                                        \
    } while (0)

#define BIS_REQUIRE(cond, ...)                                                 \
    do {                                                                       \
        if (!(cond)) {                                                         \
            bis_set_error(__VA_ARGS__);                                        \
            return 2;                                                          \
        }                                                                      \
    } while (0)

#define BIS_LAUNCH_CHECK(ctx)                                                  \
    do {                                                                       \
        if (!(ctx)->capturing) (ctx)->launches++; /* recorded launches count when replayed */ \
        cudaError_t _e = cudaGetLastError();                                   \
        if (_e != cudaSuccess) {                                               \
            bis_set_error("%s:%d: kernel launch failed: %s", __FILE__,         \
                          __LINE__, cudaGetErrorString(_e));                   \
            return 1;                                                          \
        }                                                                      \
    } while (0)

// ---- reductions -----------------------------------------------------------
// Deterministic AND partition-invariant reductions (SURVEY.md 8(e) "cross-P reproducibility").
//
// The global rows are cut into BIS_NSLAB = 8 fixed "virtual slabs" (bis_partition_rule: the 8-GPU row
// blocks); a rank of a P-GPU run (P | 8) owns 8/P consecutive slabs.  Every reducing kernel maps its
// blocks onto rows by a rule that depends on the GLOBAL problem only (streaming kernels: block b <->
// rows [b*chunk, (b+1)*chunk) of the global index space; windowed SpMV: CTA b of a fixed logical grid
// <-> positions b, b+G, ... of the slab's tile order), so a block partial is the same number at
// every rank count.  The last block to arrive adds the partials of each local slab in a fixed order
// (lane l: partials l, l+32, ... then a shuffle tree), the 8 slab sums are exchanged through the peer
// banks, and every rank adds ((s0+s1)+(s2+s3))+((s4+s5)+(s6+s7)): residual histories are bit-identical
// at 1, 2, 4 and 8 GPUs.  Where the conditions do not hold (rank count not dividing 8, a caller's own
// unaligned row blocks, the vector-CRS / TMA-gather SpMV variants) a rank contributes ONE record and
// the records are added in rank order: deterministic for a given rank count, as in round 1.
constexpr int BIS_MAX_RED_BLOCKS = 32768;  // partials per quantity
constexpr int BIS_MAX_RED = 2;             // quantities per kernel
constexpr int BIS_MAX_PEERS = 8;           // ranks a peer-memory link can span (one NVSwitch box)
constexpr int BIS_NSLAB = 8;               // virtual slabs
constexpr int BIS_RED_CHUNK_MIN = 1024;    // rows per block of a reducing streaming kernel (x 2^k)

// Peer-memory link (bis_dist.cu): every rank owns a small "bank" that all other ranks of the
// box map through CUDA IPC.  Dot products are summed over ranks by the last block of the
// reducing kernel itself (it stores its slab sums into every peer's bank over NVLink and adds
// the 8 records in the fixed order), and halo values are stored straight into the
// neighbour's ghost buffer by the pack kernel: no NCCL call on the iteration path.
// Bank layout, in doubles: [0, 2*8*4) reduction records {v0, v1, epoch, -} indexed by
// (epoch parity, record index); BIS_BANK_HALO_FLAG + s: newest halo epoch whose values from
// source s have landed; BIS_BANK_HALO_ACK + q: rank q has finished every SpMV before that epoch.
constexpr int BIS_BANK_HALO_FLAG = 256;
constexpr int BIS_BANK_HALO_ACK = 320;
constexpr size_t BIS_BANK_BYTES = (size_t)2 << 20;

struct RedArgs {
    double *partials;        // [BIS_MAX_RED][BIS_MAX_RED_BLOCKS]
    unsigned int *counter;   // ticket, self-resetting
    double *scalars;         // device scalar bank
    int slot[BIS_MAX_RED];   // target slots (-1: unused)
    int block_offset;        // first partial index written by this launch
    int total_blocks;        // partials to add when finalising
    int finalize;            // 0: only write partials (a later launch finalises)
    // local slabs: slab i covers partials [slab_off[i], slab_off[i+1])
    int n_slab;
    int slab_off[BIS_NSLAB + 1];
    // records: n_rec numbers are added in the fixed order; this rank produces [rec_first, rec_first + n_slab)
    int n_rec;
    int rec_first;
    // sum over ranks through peer memory (peer_n > 1), done by the finalising block
    int peer_n;
    int peer_rank;
    unsigned long long peer_epoch;
    double *peer_bank[BIS_MAX_PEERS];
    int *errflag;
    unsigned long long *waitstat;   // [0] ns spent waiting for the other ranks' records, [1] reductions counted
};

// How the rows of the current problem are cut (set when a matrix is created; streaming kernels of
// another length fall back to the default rule for that length).
struct RowPartition {
    int64_t n_global = 0;
    int64_t row_begin = 0;
    int64_t n_local = 0;
    int chunk = BIS_RED_CHUNK_MIN;     // rows per block of a reducing streaming kernel
    int n_slab = 1;                    // local virtual slabs (0 < n_slab <= 8)
    int slab_first = 0;                // global index of the first local slab
    int64_t slab_row[BIS_NSLAB + 1] = {};   // LOCAL row offsets of the local slab boundaries
    bool invariant = false;            // the conditions of the partition-invariant sum hold
};

// Optional per-kernel-family device timing (bis_profile_enable): cudaEvent pairs
// recorded on the launching stream around every launch of the family.
enum { BIS_PROF_SPMV = 0, BIS_PROF_SPTRSV = 1, BIS_PROF_VECTOR = 2, BIS_PROF_NTAGS = 3 };
struct ProfTag {
    std::vector<cudaEvent_t> ev;   // pairs: [2i] start, [2i+1] stop
    size_t used = 0;               // events recorded since the last flush
    double acc_ms = 0.0;
    int64_t count = 0;
};

struct bis_context {
    int device = 0;
    int rank = 0;
    int nranks = 1;
    int sm_count = 148;
    size_t l2_bytes = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t comm_stream = nullptr;
    cudaEvent_t ev_timer0 = nullptr, ev_timer1 = nullptr;
    cudaEvent_t ev_main = nullptr, ev_comm = nullptr, ev_scalar = nullptr;
    double *d_scalars = nullptr;         // BIS_NUM_SCALARS
    double *h_scalars = nullptr;         // pinned staging
    double *d_partials = nullptr;
    double *d_block_partials = nullptr;  // [2*BIS_BLOCK_MAX_K][BIS_MAX_RED_BLOCKS]: multi-RHS reductions (bis_block.cu), on first use
    unsigned int *d_counter = nullptr;
    int *d_errflag = nullptr;            // set by kernels on watchdog expiry
    void *d_flush = nullptr;
    size_t flush_bytes = 0;
    ncclComm_t comm = nullptr;           // reductions (main stream)
    ncclComm_t comm_halo = nullptr;      // halo exchange (comm stream)
    // peer-memory link (nranks <= BIS_MAX_PEERS on one box); NCCL stays as the fallback transport
    int peer_on = 0;
    double *d_bank = nullptr;                       // this rank's bank (BIS_BANK_BYTES)
    double *peer_bank[BIS_MAX_PEERS] = {};          // every rank's bank as mapped here
    unsigned long long red_epoch = 0;               // finalised reductions so far (same on all ranks)
    unsigned long long halo_epoch = 0;              // halo exchanges so far (same on all ranks)
    unsigned int *d_pack_ticket = nullptr;
    unsigned long long *d_waitstat = nullptr;       // in-kernel wait accounting (bis_dist_wait_read)
    int *d_barrier_word = nullptr;                  // operand of bis_dist_stream_barrier (always 0)
    std::vector<void *> ipc_opened;                 // mappings to close
    RowPartition part;                              // bis_partition_set (bis_context.cu)
    // CUDA graphs (bis_graph_*): `capturing` while the stream records; graph_epoch counts captures and
    // replays -- host-side knowledge about device buffers that a replay may have changed (the working
    // vectors of the triangular solves) is only trusted within one epoch
    int capturing = 0;
    uint64_t graph_epoch = 0;
    int64_t launches = 0;
    int64_t wave_solves = 0;    // triangular solves that ran as variant 5 (bis_sptrsv_wave.cuh)
    int64_t chain_solves = 0;   // triangular solves that ran as variant 4 (bis_sptrsv_chain.cuh)
    // options
    // freed vectors are kept for the next allocation of the same size (a solver allocates ~20 vectors of
    // one length; cudaMalloc + cudaFree of a gigabyte each is milliseconds); emptied when memory runs short
    std::vector<std::pair<size_t, void *>> vec_cache;
    size_t vec_cache_bytes = 0;
    std::unordered_map<void *, size_t> vec_bytes;   // live vectors of bis_vector_alloc
    int opt_vector_cache = 1;
    int opt_spmv_fused = 1;     // distributed SpMV over peer memory as ONE kernel (0: pack / interior / wait / strips launches)
    int opt_dist_p2p = 1;       // 0: NCCL transport even when the peer-memory link is up
    int opt_factor_keep_crs = 1;       // 0: a triangular factor gives up its natural-order CRS once its level-ordered copy exists
    int opt_perm_mode = 0;             // the reference's PERM_MODE: 0 NONE, 1 C (multicolouring), 2 BFS, 3 RCM, 4 CM; read by the host's preprocessing
    int opt_precond_inner_iters = 0;   // PRECOND_INNER_ITERS of the reference (kernels.hpp:321): inner sweeps of -p 2st / s2st
    int opt_graph = 1;          // the host stack records iteration bodies as CUDA graphs (bis_context_get_option)
    int opt_spmv_variant = 0;
    int opt_spmv_lanes = 0;
    int opt_trsv_variant = 0;
    int opt_trsv_poll_ns = 0;   // sleep between polls in the triangular solve (0: default)
    int opt_trsv_block = 256;   // triangular solve: rows per block (64, 128, 256)
    int opt_trsv_gates = 1;     // triangular solve: staged waiting on the per-row gates (0: poll all operands)
    int opt_trsv_sleep[4] = {0, 60, 250, 1000};   // ns between polls of a gate 1, 2, 3, >= 4 levels back (>= 6: twice the last)
    int opt_trsv_debug = 0;     // dump per-row timestamps of each solve to $BIS_TRSV_DEBUG_FILE
    int opt_spmv_rows = 0;      // TMA variant: rows per tile (0 auto)
    int opt_spmv_stages = 0;    // TMA variant: max stages (0 auto)
    int opt_spmv_vdict = 1;     // windowed SpMV: 1 = stream 1-byte value indices when the matrix has <= 256 distinct values (lossless,
                                // + 1 byte per nonzero of memory; 0 = stream the values; see DESIGN.md 3.1)
    int last_spmv_value_bytes = 8;   // bytes per nonzero the last windowed SpMV streamed for the values (8 or 1)
    int64_t last_spmv_stream_bytes = 0;   // compulsory HBM bytes of the last windowed SpMV launch (its format's byte model)
    int opt_wave_cluster = 8;   // stencil wavefront: planes per thread-block cluster (1: no clusters, every hand-over through L2)
    int opt_wave_backoff_ns = 0;      // ... nanoseconds a plane fed through L2 falls back after it had to poll (clusters only)
    int wave_cluster_used = 0;  // ... what the last solve ran with
    int opt_wave_debug = 0;     // stencil-wavefront perf experiments (results invalid); only in -DBIS_PERF_DEBUG builds
    int opt_spmv_debug = 0;     // perf experiments (results invalid when non-zero); only in -DBIS_PERF_DEBUG builds
    int opt_win_rows = 0;       // variant 3: rows per tile (0 auto; fixed once a matrix's format is built)
    int opt_spmv_mult = 0;      // TMA variant: threads per tile row (1, 2, 4; 0 auto)
    int opt_spmv_blocked = 0;   // TMA variant: 1 = contiguous tile run per CTA instead of interleaved
    int opt_spmv_smem_kb = 0;   // TMA variant: shared-memory budget per CTA (0 auto)
    int opt_spmv_l2_mb = 0;     // variant 3: matrix bytes streamed between two uses of an x plane above which the sweep is y-blocked (0: 40 MB)
    int profile = 0;
    ProfTag prof[BIS_PROF_NTAGS];
    // cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute: remembered per context
    std::unordered_map<const void *, size_t> smem_configured;
};

// Variant 4 of the triangular solve (bis_sptrsv_chain.cuh): sliced-ELL records of 32 chains per warp
struct ChainFormat {
    int state = 0;                 // 0 not built, 1 usable, -1 not representable (fall back to the dataflow solve)
    int K = 0;                     // nonzeros per record row (max row length)
    int n_groups = 0;              // warps
    long long n_recs = 0;          // warp steps over all groups
    unsigned char *d_recs = nullptr;
    long long *d_slice_off = nullptr;   // [n_groups + 1]
    double *d_w = nullptr;              // [32 * n_recs] working vector, record-major
};

// Variant 5 of the triangular solve (bis_sptrsv_wave.cuh): records of a structured-grid factor
struct WaveFormat {
    int state = 0;                 // 0 not tried, 1 usable, -1 not a (<= 27-point) stencil in natural ordering
    int nx = 0, ny = 0, nz = 0, W = 0, S = 0;
    long long n_groups = 0;
    double *d_rec = nullptr;       // [n_groups][S][13][32]
    double *d_w[2] = {nullptr, nullptr};   // working vectors [n_groups][S][32]; solves alternate, each re-arms the other
    int w_clean[2] = {0, 0};
    uint64_t w_epoch = 0;
    int w_cluster = 0;             // cluster size of the solves that left the working vectors in their present state
    unsigned int *d_ticket = nullptr;
    int cluster_fit[17] = {-1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1};   // clusters of that many CTAs the device holds at once (-1: not asked yet)
};

struct LevelSets {
    bool built = false;            // level analysis done (skipped while the stencil wavefront serves the factor)
    mutable WaveFormat wave;
    int n_levels = 0;
    int64_t n_slots = 0;              // == n_rows: position in the level-ordered row list
    int *d_slot_row = nullptr;        // [n_slots] original row
    int *d_level = nullptr;           // [n_rows] level of every row (kept for the chain format)
    mutable ChainFormat chain;
    int *d_slot_level = nullptr;      // [n_slots] level of that row (non-decreasing)
    int *d_slot_gate = nullptr;       // [4*n_slots] three gate columns + their packed level distances (bis_matrix.cu)
    int *d_level_size = nullptr;      // [n_levels] rows per level
    std::vector<int64_t> level_start; // [n_levels+1] host copy (per-level launch variant)
    unsigned int *d_level_done = nullptr;   // [n_levels] completion counters
    unsigned int *d_ticket = nullptr; // chunk ticket
    double *d_w = nullptr;            // [n_slots] working vector of the solve IN SLOT ORDER: sentinel until the slot's value is final
    double *d_w2 = nullptr;           // its twin: solves alternate between the two, each resets the other one while it runs
    int w_clean[2] = {1, 1};          // host's knowledge: that working vector holds "not ready" everywhere
    uint64_t w_epoch = 0;             // ... valid while the context's graph_epoch has this value
    // level-ordered copy of the strict factor (rows stored in slot order, operands named by slot)
    int64_t *d_rp = nullptr;          // [n_slots+1]
    int *d_col = nullptr;
    double *d_val = nullptr;
};

// entry points that read a matrix's natural-order CRS arrays
#define BIS_REQUIRE_CRS(A) BIS_REQUIRE(!(A)->crs_released, "this factor gave up its natural-order CRS arrays (option factor_keep_crs = 0): only triangular solves can use it")

struct HaloPlan {
    int64_t n_ghost = 0;                 // ghost elements appended after owned
    double *d_ghost = nullptr;           // [n_ghost] received values
    double *d_sendbuf = nullptr;         // [n_send]
    int *d_send_idx = nullptr;           // [n_send] local row indices to pack
    int *d_ghost_global = nullptr;       // [n_ghost] global column id of each ghost (sorted)
    int64_t n_send = 0;
    std::vector<int64_t> recv_off;       // [nranks+1] segments of d_ghost
    std::vector<int64_t> send_off;       // [nranks+1] segments of d_sendbuf
    int64_t interior_begin = 0, interior_end = 0;   // rows without ghosts
    // peer-memory transport: d_ghost holds two copies (epoch parity), ghost_stride doubles apart
    int64_t ghost_stride = 0;
    mutable const double *cur_ghost = nullptr;      // the copy the current SpMV reads
    double *peer_ghost[BIS_MAX_PEERS] = {};         // rank p's d_ghost as mapped here
    std::vector<int64_t> peer_recv_off;             // [nranks] where my values start in rank p's ghost list
    std::vector<int64_t> peer_stride;               // [nranks] rank p's ghost_stride
    bool peer_ready = false;
};

// Kernel arguments of the fused distributed SpMV (bis_spmv_win.cuh); filled by bis_halo_fuse_args (bis_dist.cu)
struct HaloFuse {
    int n_dst, n_src, n_ranks, me;
    int dst_rank[BIS_MAX_PEERS], src_rank[BIS_MAX_PEERS];
    int64_t seg_off[BIS_MAX_PEERS + 1];            // segments of the send list, one per destination
    double *dst[BIS_MAX_PEERS];                    // where that segment lands in the destination's ghost copy
    unsigned long long *dst_flag[BIS_MAX_PEERS];   // destination's bank: HALO_FLAG + me
    unsigned long long *ack_out[BIS_MAX_PEERS];    // rank p's bank: HALO_ACK + me
    const unsigned long long *ack_in;              // my bank: HALO_ACK
    const unsigned long long *flag_in;             // my bank: HALO_FLAG
    const int *send_idx;
    unsigned int *ticket;
    unsigned long long epoch;
    int *errflag;
    unsigned long long *waitstat;   // [2] ns CTA 0's producer waited for the senders' flags, [3] exchanges counted
};

// Acceleration structure of SpMV variant 3 (bis_spmv_win.cuh), derived lazily from the CRS arrays.
struct WinFormat {
    int state = 0;                 // 0 not built, 1 usable, -1 not representable (fall back)
    int R = 0;                     // rows per tile
    int cap = 0;                   // nonzeros per stage
    int xcap = 0;                  // x-window doubles per stage
    int64_t n_tiles = 0;
    int *d_seg_start = nullptr;
    unsigned short *d_seg_len = nullptr;
    unsigned short *d_seg_off = nullptr;
    int *d_nseg = nullptr;
    unsigned short *d_lidx = nullptr;
    // value dictionary (lossless): when the matrix holds at most 256 distinct values (constant-coefficient stencils:
    // HPCG has two), the tiles stream a 1-byte index per nonzero instead of the 8-byte value and the kernel looks the
    // value up in a 2 KB table in shared memory -- the bits of every product are those of the CRS value
    int dict_state = 0;            // 0 not tried, 1 usable, -1 more than 256 distinct values (or switched off)
    int n_dict = 0;
    unsigned char *d_vidx = nullptr;   // [nnz + 32]
    double *d_vdict = nullptr;         // [256], ascending bit patterns
    // processing order of the tiles (bis_spmv.cu: win_build_order)
    int *d_order = nullptr;        // [n_tiles]; bit 31: the tile reads ghosts
    int n_slab = 1;                // local virtual slabs the order is cut into
    int pos0[BIS_NSLAB + 1] = {};  // positions of slab i: [pos0[i], pos0[i+1])
    bool invariant = false;        // per-(slab, CTA) partials are partition-invariant
    int slab_first = 0;
    int traversal_blocks = 1;      // y-blocks of the interior traversal (1: natural order)
};

struct bis_matrix {
    int64_t n_rows = 0;        // local rows
    int64_t n_cols = 0;        // local owned columns (== n_rows when square)
    int64_t n_rows_global = 0;
    int64_t row_begin = 0;     // first global row
    int64_t nnz = 0;           // local nnz
    int64_t nnz_global = 0;
    int rp_bytes = 4;          // 4 or 8
    void *d_rp = nullptr;      // int32_t or int64_t [n_rows+1]
    int *d_col = nullptr;      // local column ids (ghosts >= n_cols)
    double *d_val = nullptr;
    int triangular = 0;        // 0 general, 1 strictly lower, 2 strictly upper
    int64_t grid_nx = 0, grid_ny = 0, grid_nz = 0;   // structured-grid hint of the generators (0: unknown)
    double mean_row = 0.0;
    int max_row = 0;
    mutable LevelSets lv;
    HaloPlan halo;
    mutable WinFormat win;
    bool distributed = false;
    bool crs_released = false; // triangular factor whose natural-order d_rp / d_col / d_val were freed (option factor_keep_crs = 0)
};

// ---- internal entry points shared between translation units ---------------
int bis_reduce_finish(bis_context *ctx, int slot_a, int slot_b);
RedArgs bis_red_args(bis_context *ctx, int slot_a, int slot_b);
void bis_red_set_slabs(const bis_context *ctx, RedArgs &ra, const RowPartition &part, const int *off, int total);
// 8 virtual slabs of a problem: vb[0..8] global row boundaries, *chunk rows per reducing block
void bis_partition_rule(int64_t n_global, int64_t plane, int64_t vb[BIS_NSLAB + 1], int *chunk);
// the row block of `rank` under that rule (unions of virtual slabs when nranks divides 8)
void bis_partition_rows(int64_t n_global, int64_t plane, int rank, int nranks, int64_t *begin, int64_t *end);
// records the partition of the matrix just created (plane = 0: no plane structure known)
void bis_partition_set(bis_context *ctx, int64_t n_global, int64_t plane, int64_t row_begin, int64_t n_local);
// partition to use for a streaming kernel over n local rows
RowPartition bis_partition_for(const bis_context *ctx, int64_t n);
int bis_halo_exchange_begin(bis_context *ctx, const bis_matrix *A, const double *x);
int bis_halo_exchange_end(bis_context *ctx, const bis_matrix *A);
// starts a halo exchange that the SpMV kernel itself performs: advances the epoch, selects the ghost copy
int bis_halo_fuse_args(bis_context *ctx, const bis_matrix *A, HaloFuse *hf);
int bis_peer_link_setup(bis_context *ctx);
void bis_peer_link_teardown(bis_context *ctx);
// maps a cudaMalloc'ed buffer of every rank into this process (collective); out[p] for p == rank is `mine`
int bis_peer_map(bis_context *ctx, void *mine, void **out);
int bis_matrix_finalize_distributed(bis_context *ctx, bis_matrix *A,
                                    int *d_col_global_in_place);
int bis_build_levels_device(bis_context *ctx, bis_matrix *T);
// the level sets of a factor that has been served by the stencil wavefront so far (bis_factor.cu)
int bis_ensure_levels(bis_context *ctx, const bis_matrix *T);
// the values of A changed in place (bis_matrix_scale_symmetric): the SpMV's value dictionary is rebuilt on next use (bis_spmv.cu)
void bis_win_values_changed(const bis_matrix *A);
// tries to build the stencil-wavefront records of a triangular factor (bis_sptrsv.cu); wave.state tells
int bis_wave_build(bis_context *ctx, const bis_matrix *T);
int bis_matrix_stats(bis_context *ctx, bis_matrix *A);
// builds the SpMV acceleration structure of a general matrix (bis_spmv.cu); lazy on first SpMV otherwise
int bis_spmv_prepare(bis_context *ctx, const bis_matrix *A);
// raises the dynamic shared memory limit of `func` on the context's device when it is below `bytes`
int bis_ensure_dynamic_smem(bis_context *ctx, const void *func, size_t bytes);
int bis_prof_begin(bis_context *ctx, int tag);
int bis_prof_end(bis_context *ctx, int tag);

// cudaMalloc that empties the contexts' vector caches and retries once when the device is out of memory
void bis_vector_cache_release_all();
void bis_vector_cache_trim(bis_context *ctx);
template <typename T> static inline cudaError_t bis_cuda_malloc(T **p, size_t bytes) {
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(p), bytes);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        bis_vector_cache_release_all();
        e = cudaMalloc(reinterpret_cast<void **>(p), bytes);
    }
    return e;
}

// NVTX ranges named like the reference's LIKWID regions (kernels.hpp:25-40,56-75,90-106): "spmv",
// "sptrsv", "backwards-sptrsv".  Without an attached tool a push/pop is a null-pointer check.
struct BisNvtxRange {
    explicit BisNvtxRange(const char *name) { nvtxRangePushA(name); }
    ~BisNvtxRange() { nvtxRangePop(); }
    BisNvtxRange(const BisNvtxRange &) = delete;
    BisNvtxRange &operator=(const BisNvtxRange &) = delete;
};

static inline int bis_blocks_for(int64_t n, int per_block, int cap) {
    int64_t b = (n + per_block - 1) / per_block;
    if (b < 1) b = 1;
    if (b > cap) b = cap;
    return (int)b;
}
