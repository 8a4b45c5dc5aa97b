/* bis_b200.h -- C-ABI of the B200-native (sm_100a) iteration-loop hot path of
 * DanecLacey/basic_iterative_solvers.
 *
 * This header is the drop-in boundary (SURVEY.md 8(b)).  Every entry point
 * cites the reference interface it replaces as file:line under the reference
 * tree.  Conventions:
 *
 *  - plain C: opaque handles, raw pointers, sizes; no C++ or torch types.
 *  - every function returns 0 on success, non-zero on failure; the message is
 *    available from bis_last_error() (thread-local).  There is NO CPU
 *    fallback: without a usable CUDA device every call fails.
 *  - `double *` arguments marked [dev] are DEVICE addresses obtained from
 *    bis_vector_alloc().  They are ordinary addresses: the host may offset
 *    them (&V[j*N], methods/gmres.hpp:168) and swap them (std::swap,
 *    methods/cg.hpp:129-133) exactly as the reference does with host
 *    pointers.  [host] marks host memory; it is never retained after the
 *    call returns.
 *  - all work is enqueued on the context's stream; only calls that return a
 *    value to [host] memory synchronise.
 *  - a context is not thread-safe (the reference harness is single-threaded,
 *    solver_harness.hpp:7-61).
 *  - in a distributed context (bis_context_create_distributed) matrices are
 *    row-partitioned, vectors hold the local rows; halo values and the
 *    partial sums of reductions move over peer memory (CUDA IPC mappings,
 *    NVLink stores issued from inside the SpMV / reducing kernels).  NCCL
 *    sets the link up and is the fallback transport (option "dist_p2p" = 0).
 *    Reductions add 8 fixed slab sums in a fixed order: bit-identical
 *    results at 1, 2, 4 and 8 GPUs (bis_partition_row_block).
 */
#ifndef BIS_B200_H
#define BIS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BIS_VERSION 100

typedef struct bis_context bis_context;
typedef struct bis_matrix bis_matrix;

/* PrecondType, common.hpp:38-47 (same order, same values) */
enum {
    BIS_PRECOND_NONE = 0,
    BIS_PRECOND_JACOBI = 1,
    BIS_PRECOND_GS = 2,
    BIS_PRECOND_BGS = 3,
    BIS_PRECOND_SGS = 4,
    BIS_PRECOND_2ST = 5,
    BIS_PRECOND_S2ST = 6,
    BIS_PRECOND_ILU0 = 7
};

/* Number of device-resident scalar slots per context (see "device scalars"). */
#define BIS_NUM_SCALARS 128

/* ---- errors / info ------------------------------------------------------ */
const char *bis_last_error(void);
int bis_version(void);
int bis_device_count(int *count);

/* ---- context ------------------------------------------------------------ */
/* Replaces: nothing in the reference (it has no device); plays the role of the
 * `Interface *smax` handle threaded through every kernel call
 * (common.hpp:14-24, kernels.hpp:44-46). */
int bis_context_create(int device, bis_context **ctx);
/* One process per GPU.  nccl_id: the 128-byte ncclUniqueId produced by
 * bis_nccl_unique_id() on rank 0 and broadcast by the caller (e.g. with
 * torch.distributed).  New in the build: the reference is single-process
 * (sparse_matrix.hpp:654-656 splits into 1 piece). */
int bis_context_create_distributed(int device, int rank, int nranks,
                                   const void *nccl_id, size_t nccl_id_bytes,
                                   bis_context **ctx);
int bis_nccl_unique_id(void *out, size_t bytes);
int bis_context_destroy(bis_context *ctx);
int bis_context_synchronize(bis_context *ctx);
int bis_context_rank(const bis_context *ctx, int *rank, int *nranks);
/* info[0]=SM count, info[1]=free bytes, info[2]=total bytes, info[3]=kernel
 * launches issued by this context so far, info[4]=L2 bytes, info[5]=1 when
 * the reductions and halo exchanges of a distributed context run over peer
 * memory (CUDA IPC + NVLink stores inside the kernels), 0 when over NCCL,
 * info[6]=triangular solves that ran as the chain variant (trsv_variant 4) */
int bis_context_info(bis_context *ctx, int64_t info[8]);
/* Device timing on the context's stream (cudaEvent pair). */
int bis_timer_start(bis_context *ctx);
int bis_timer_stop(bis_context *ctx, double *elapsed_ms /* [host] */);
/* Per-kernel-family device timing: cudaEvent pairs on the context's stream
 * around every launch of the family ("spmv", "sptrsv", "vector").  Replaces
 * the TIME(timers->spmv, ...) stopwatches and LIKWID regions of the reference
 * (common.hpp:249-254, kernels.hpp:25-40), which cannot see asynchronous
 * device work.  enable(on) resets the accumulators; read synchronises. */
int bis_profile_enable(bis_context *ctx, int on);
int bis_profile_read(bis_context *ctx, const char *family,
                     double *total_ms /* [host] */, int64_t *launches /* [host] */);
/* Write `bytes` of scratch to evict L2 between timed launches. */
int bis_flush_l2(bis_context *ctx);
/* Tuning knobs (all have defaults): key = "spmv_variant" (0 auto, 1 vector
 * CRS, 2 TMA-staged tiles + gathers, 3 windowed x), "spmv_lanes" (0 auto,
 * 2..32), "trsv_variant" (0 auto, 1 launch per level, 2 level counters,
 * 3 dataflow, 4 chains, 5 stencil wavefront), "spmv_vdict" (default 0; 1: the
 * windowed SpMV of a matrix with at most 256 distinct values streams a 1-byte
 * index per nonzero instead of the 8-byte value -- lossless, same bits;
 * "spmv_value_bytes" reads back what the last launch streamed), "wave_cluster" (stencil
 * wavefront: planes per thread-block cluster, 1 / 2 / 4 / 8 (default) / 16;
 * 1 = every plane-to-plane hand-over through L2), "perm_mode" (0 none,
 * 1 multicolouring, 2 BFS levels, 3 reverse Cuthill-McKee, 4 Cuthill-McKee:
 * read by the host's preprocessing), "graph" (0/1: the host stack
 * replays the iteration body as a CUDA graph; default 1 on one GPU),
 * "factor_keep_crs" (default 1; 0: bis_matrix_split_triangular / bis_matrix_ilu0
 * return factors that keep only their level-ordered copy -- bis_sptrsv /
 * bis_bsptrsv / bis_apply_preconditioner(gs, bgs, sgs, ilu0) work, every entry
 * point that reads the factor's CRS arrays fails loudly; the C++ host asks for
 * it when a Krylov method uses the factors in such a preconditioner only),
 * "spmv_fused", "dist_p2p", "vector_cache", ... (bis_context.cu). */
int bis_context_set_option(bis_context *ctx, const char *key, int value);
int bis_context_get_option(bis_context *ctx, const char *key, int *value /* [host] */);

/* ---- CUDA graphs --------------------------------------------------------
 * New in the build (SURVEY.md section 7 step 8).  The body of an iteration
 * (methods/cg.hpp:6-54, bicgstab.hpp:8-83, gmres.hpp:150-183, ...) is a fixed
 * sequence of launches whose scalars live on the device: between begin and
 * end the ordinary calls of this header are RECORDED instead of executed
 * (only enqueue-type calls are allowed: no upload/download, no scalar read,
 * no matrix creation), launch replays the recording.  Results are bit-
 * identical to issuing the calls.  Single-GPU contexts only. */
typedef struct bis_graph bis_graph;
int bis_graph_begin(bis_context *ctx);
int bis_graph_end(bis_context *ctx, bis_graph **graph /* out */);
int bis_graph_abort(bis_context *ctx);
int bis_graph_launch(bis_context *ctx, bis_graph *graph);
int bis_graph_free(bis_context *ctx, bis_graph *graph);
/* Row block [begin, end) of `rank` in an n_global-row problem split over `nranks` GPUs: the rule the
 * generators use (unions of 8 fixed virtual slabs when nranks divides 8, so that reductions add the
 * same partial sums in the same order at 1, 2, 4 and 8 GPUs; `plane` = rows per grid plane or 0, only
 * used for rank counts that do not divide 8).  Pure function, no device needed.  New in the build:
 * the reference is single-process (SURVEY.md F2). */
/* In-kernel wait accounting of a distributed context, in ns: out[0] time the finalising blocks of
 * reductions waited for the other ranks' records, out[1] reductions counted, out[2] time the fused
 * SpMV's first producer warp waited for the senders' halo flags, out[3] exchanges counted. */
int bis_dist_wait_read(bis_context *ctx, double out[4] /* [host] */, int reset);
/* Measurement aid: everything enqueued on the context's stream after this call starts only when every rank's
 * stream has reached it (no-op on a single-GPU context).  Used to open a timed region on all ranks together. */
int bis_dist_stream_barrier(bis_context *ctx);
int bis_partition_row_block(int64_t n_global, int64_t plane, int rank, int nranks,
                            int64_t *begin /* [host] */, int64_t *end /* [host] */);

/* ---- vectors ------------------------------------------------------------ */
/* Replaces `new double[N]` / `delete[]` in Solver::allocate_structs and the
 * destructors (solver.hpp:82-145 and the per-method overrides). */
int bis_vector_alloc(bis_context *ctx, int64_t n, double **v /* out [dev] */);
int bis_vector_free(bis_context *ctx, double *v /* [dev] */);
int bis_vector_upload(bis_context *ctx, double *dst /* [dev] */,
                      const double *src /* [host] */, int64_t n);
int bis_vector_download(bis_context *ctx, double *dst /* [host] */,
                        const double *src /* [dev] */, int64_t n);

/* ---- matrices ----------------------------------------------------------- */
/* Device mirror of MatrixCRS (sparse_matrix.hpp:59-179): row_ptr/col/val
 * copied to HBM in the order given (within-row order is preserved: it fixes
 * the summation order, SURVEY.md F9).  In a distributed context the arrays
 * are the caller's LOCAL rows [row_begin, row_begin+n_rows) with GLOBAL
 * column indices; halo index lists are derived here. */
int bis_matrix_upload_crs(bis_context *ctx, int64_t n_rows, int64_t n_cols,
                          int64_t nnz, const int32_t *row_ptr /* [host] */,
                          const int32_t *col /* [host] */,
                          const double *val /* [host] */, bis_matrix **A);
/* 64-bit row_ptr (the reference's `int nnz` cannot hold HPCG-512, F5). */
int bis_matrix_upload_crs64(bis_context *ctx, int64_t n_rows, int64_t n_cols,
                            int64_t nnz, const int64_t *row_ptr /* [host] */,
                            const int32_t *col /* [host] */,
                            const double *val /* [host] */, bis_matrix **A);
/* convert_coo_to_crs (utilities/utilities.hpp:326-367) together with the reader's stable sort by row
 * (sparse_matrix.hpp:20-30, 332-344), on the device: entries in any order (sorted = 0) or already grouped
 * by row (sorted != 0, the reference's is_sorted); inside a row they keep their order of appearance,
 * which is the summation order of every kernel.  0-based indices. */
int bis_matrix_upload_coo(bis_context *ctx, int64_t n_rows, int64_t n_cols, int64_t nnz,
                          const int32_t *I /* [host] */, const int32_t *J /* [host] */,
                          const double *V /* [host] */, int sorted, bis_matrix **A /* out */);
int bis_matrix_upload_crs_distributed(bis_context *ctx, int64_t row_begin,
                                      int64_t n_rows_local,
                                      int64_t n_rows_global, int64_t nnz_local,
                                      const int64_t *row_ptr /* [host] */,
                                      const int32_t *col /* [host], global */,
                                      const double *val /* [host] */,
                                      bis_matrix **A);
/* Strictly triangular factor (L_strict / U_strict of split_LU_new,
 * utilities/LU_factors.hpp:122-309, or of factor_ILU0_old, :320-539) plus the
 * level sets the level-scheduled solves need.  upper != 0 for U_strict. */
int bis_matrix_upload_triangular(bis_context *ctx, int64_t n, int64_t nnz,
                                 const int32_t *row_ptr /* [host] */,
                                 const int32_t *col /* [host] */,
                                 const double *val /* [host] */, int upper,
                                 bis_matrix **T);
/* Device-side synthetic generators (SURVEY.md 8(d)); in a distributed context
 * each rank generates its own contiguous slab of rows.  Replaces the
 * .mtx/SCAMAC input path (main.cpp:47-58) for sizes the reference cannot
 * hold. */
int bis_matrix_generate_hpcg(bis_context *ctx, int nx, int ny, int nz,
                             bis_matrix **A);
int bis_matrix_generate_anderson(bis_context *ctx, int lx, int ly, int lz,
                                 double ranpot, double t, uint64_t seed,
                                 int periodic, bis_matrix **A);
int bis_matrix_free(bis_context *ctx, bis_matrix *A);
/* info[0]=local rows, [1]=global rows, [2]=local nnz, [3]=global nnz,
 * [4]=row_ptr bytes per entry, [5]=number of levels (triangular),
 * [6]=halo elements received per SpMV, [7]=first global row */
int bis_matrix_info(const bis_matrix *A, int64_t info[8]);
/* Copy the (local) device CRS back (tests compare generators with numpy). */
int bis_matrix_download_crs(bis_context *ctx, const bis_matrix *A,
                            int64_t *row_ptr /* [host] n+1 */,
                            int32_t *col /* [host] nnz, global ids */,
                            double *val /* [host] nnz */);
/* D[r] = A[r][r] (peel_diag_crs_new's D output, LU_factors.hpp:827-869),
 * D_inv optional. */
int bis_matrix_extract_diagonal(bis_context *ctx, const bis_matrix *A,
                                double *D /* [dev] */,
                                double *D_inv /* [dev] or NULL */);
/* -scale: A <- D^-1/2 A D^-1/2 in place with D_scale[r] = 1/sqrt(|A[r][r]|)
 * (extract_scale + scale_mat, LU_factors.hpp:880-898, preprocessing.hpp:15-24;
 * 0.0 for a row without diagonal as solver.hpp:105 leaves it, fatal on a zero
 * diagonal).  D_scale is written; the caller scales b and x_0 with it
 * (preprocessing.hpp:48-49).  Distributed matrices fetch the factors of their
 * ghost columns from the owners. */
int bis_matrix_scale_symmetric(bis_context *ctx, bis_matrix *A,
                               double *D_scale /* [dev] out */);

/* ---- permutation seam ---------------------------------------------------
 * The reference permutes A, b and x_0 before factoring when built with SMAX and a PERM_MODE other than NONE
 * (preprocessing.hpp:52-65; generate_perm / apply_mat_perm / apply_vec_perm, utilities/smax_helpers.hpp:44-80;
 * modes RS, BFS, C, ...: CMakeLists.txt:129-133).  SMAX is absent, so this is a LABELLED mode of the build with
 * its own fixtures (option "perm_mode" = 1, the reference's PERM_MODE = C "colouring"): rows ordered by
 * (colour, row) of a multicolouring of A's graph -- a triangular factor of P A P^T has one level per colour.
 * Iteration counts differ from the unpermuted solve; x_star stays in the permuted numbering, as in the reference. */
int bis_matrix_colouring_permutation(bis_context *ctx, const bis_matrix *A, int *perm /* [dev] int32[n], perm[new] = old */,
                                     int *inv_perm /* [dev] int32[n] */, int *n_colours /* [host] */);
/* The breadth-first family of orderings (what SMAX's generate_perm offers besides colouring; smax_helpers.hpp:51-53):
 * mode 2 = rows by (BFS level, row), 3 = reverse Cuthill-McKee, 4 = Cuthill-McKee; the search starts at the row of
 * smallest degree and restarts there for every further component.  n_levels: BFS levels over all components. */
int bis_matrix_bfs_permutation(bis_context *ctx, const bis_matrix *A, int mode, int *perm /* [dev] int32[n], perm[new] = old */,
                               int *inv_perm /* [dev] int32[n] */, int *n_levels /* [host] */);
int bis_matrix_permute_symmetric(bis_context *ctx, const bis_matrix *A, const int *perm /* [dev] */,
                                 const int *inv_perm /* [dev] */, bis_matrix **B /* out: P A P^T */);
int bis_vector_permute(bis_context *ctx, double *out /* [dev] */, const double *in /* [dev] */,
                       const int *perm /* [dev] */, int64_t n);     /* out[i] = in[perm[i]] */
int bis_index_alloc(bis_context *ctx, int64_t n, int **p /* out [dev] */);
int bis_index_free(bis_context *ctx, int *p /* [dev] */);
int bis_index_download(bis_context *ctx, int32_t *dst /* [host] */, const int *src /* [dev] */, int64_t n);
/* Device split of A into strictly lower / upper triangular matrices with level
 * sets (split_LU_new, LU_factors.hpp:122-309), single-GPU contexts only. */
int bis_matrix_split_triangular(bis_context *ctx, const bis_matrix *A,
                                bis_matrix **L_strict, bis_matrix **U_strict);
/* ILU(0) of the device matrix A, on the device (factor_ILU0_old,
 * LU_factors.hpp:320-539: row-wise IKJ on A's pattern, pivots |u_kk| < 1e-16
 * skipped :370, updates only where the working value is != 0.0 :384, diagonals
 * |u_ii| < pivot_tolerance replaced by +-pivot_replacement :410-412).  Rows are
 * factored in dependency order by one launch; the result is bit-identical to
 * the sequential routine.  Returns the strict factors (columns ascending, as
 * the reference stores them) with their level sets, L_D = 1 (optional) and
 * U_D = diag(U).  Single-GPU contexts only. */
int bis_matrix_ilu0(bis_context *ctx, const bis_matrix *A,
                    double pivot_tolerance, double pivot_replacement,
                    bis_matrix **L_strict, bis_matrix **U_strict,
                    double *L_D /* [dev] or NULL */, double *U_D /* [dev] */);

/* ---- kernels.hpp seam: one entry per reference kernel ------------------- */
/* spmv / native_spmv, kernels.hpp:22-52.  x may be offset by the caller
 * (gmres.hpp:168-170 passes &V[k*N]). */
int bis_spmv(bis_context *ctx, const bis_matrix *A, const double *x /* [dev] */,
             double *y /* [dev] */);
/* sptrsv / native_sptrsv, kernels.hpp:54-86: x[r]=(b[r]-sum L*x)/D[r], rows
 * ascending; x may alias b. */
int bis_sptrsv(bis_context *ctx, const bis_matrix *L_strict, double *x,
               const double *D, const double *b);
/* bsptrsv / native_bsptrsv, kernels.hpp:88-117: rows descending. */
int bis_bsptrsv(bis_context *ctx, const bis_matrix *U_strict, double *x,
                const double *D, const double *b);
/* kernels.hpp:119-153; out may alias a or b. */
int bis_subtract_vectors(bis_context *ctx, double *out, const double *a,
                         const double *b, int64_t n, double scale);
int bis_sum_vectors(bis_context *ctx, double *out, const double *a,
                    const double *b, int64_t n, double scale);
int bis_elemwise_mult_vectors(bis_context *ctx, double *out, const double *a,
                              const double *b, int64_t n, double scale);
int bis_elemwise_div_vectors(bis_context *ctx, double *out, const double *a,
                             const double *b, int64_t n, double scale);
/* kernels.hpp:155-162 */
int bis_compute_residual(bis_context *ctx, const bis_matrix *A, const double *x,
                         const double *b, double *residual, double *tmp);
/* kernels.hpp:194-212; result to [host] (after allreduce when distributed). */
int bis_euclidean_vec_norm(bis_context *ctx, const double *v, int64_t n,
                           double *result /* [host] */);
int bis_dot(bis_context *ctx, const double *a, const double *b, int64_t n,
            double *result /* [host] */);
/* kernels.hpp:214-220, 236-241, 252-257 */
int bis_scale(bis_context *ctx, double *out, const double *v, double scalar,
              int64_t n);
int bis_init_vector(bis_context *ctx, double *v, double value, int64_t n);
int bis_copy_vector(bis_context *ctx, double *out, const double *in, int64_t n);
/* normalize_x, methods/jacobi.hpp:27-40 */
int bis_normalize_x(bis_context *ctx, double *x_new, const double *x_old,
                    const double *D, const double *b, int64_t n);
/* apply_preconditioner, kernels.hpp:336-414 (PRECOND_OUTER_ITERS = 1,
 * PRECOND_INNER_ITERS = 0).  out may alias in (gmres.hpp:173-176). */
int bis_apply_preconditioner(bis_context *ctx, int precond, int64_t n,
                             const bis_matrix *L_strict,
                             const bis_matrix *U_strict, const double *A_D,
                             const double *A_D_inv, const double *L_D,
                             const double *U_D, double *out, double *in,
                             double *tmp, double *work);

/* ---- device scalars ----------------------------------------------------- */
/* The Krylov recurrences consume dot products as scalars (alpha, beta, omega,
 * rho, h_jk).  The reference holds them in host doubles (cg.hpp:18-47); here
 * they live in BIS_NUM_SCALARS device slots so that a whole iteration can be
 * enqueued without a host round trip.  Reductions write a slot (already
 * summed over ranks in a distributed context); fused kernels read slots. */
int bis_scalar_set(bis_context *ctx, int slot, double value);
int bis_scalar_get(bis_context *ctx, int first_slot, int count,
                   double *values /* [host] */); /* synchronises */
/* Split read (the harness samples the residual norm every iteration,
 * solver_harness.hpp:24): _begin enqueues the copy behind the work queued so far
 * and returns; _end waits for that copy only, so kernels queued in between (the
 * next iteration, run ahead by the host) keep the device busy meanwhile.  One
 * read may be outstanding per context. */
int bis_scalar_read_begin(bis_context *ctx, int first_slot, int count);
int bis_scalar_read_end(bis_context *ctx, int first_slot, int count,
                        double *values /* [host] */);
int bis_scalar_copy(bis_context *ctx, int dst_slot, int src_slot);
/* slot <- sum a*b ; slot <- sum v*v (NOT the square root) */
int bis_dot_to_slot(bis_context *ctx, const double *a, const double *b,
                    int64_t n, int slot);
int bis_sumsq_to_slot(bis_context *ctx, const double *v, int64_t n, int slot);

/* ---- fused kernels (additional exports, SURVEY.md 8(b)) ----------------- */
/* Same arithmetic per element as the reference sequence they replace; only
 * memory passes and launches are merged. */

/* y = A x ; slot_yw <- (y,w) ; slot_yy <- (y,y) if slot_yy >= 0.
 * cg.hpp:16,23 (w = p_old) ; bicgstab.hpp:30,34 (w = r0) and :48,51 (w = s). */
int bis_spmv_dot(bis_context *ctx, const bis_matrix *A, const double *x,
                 double *y, const double *w, int slot_yw, int slot_yy);
/* compute_residual + squared norm: tmp = A x (stored if tmp != NULL),
 * r = b - tmp, slot_rr <- (r,r).  kernels.hpp:155-162 + :194-203, as used by
 * jacobi.hpp:102-107, gauss_seidel.hpp:99-104 and every init_residual. */
int bis_spmv_residual(bis_context *ctx, const bis_matrix *A, const double *x,
                      const double *b, double *r, double *tmp, int slot_rr);
/* Jacobi sweep: x_new = (b - (A x_old - D x_old)) / D, jacobi.hpp:27-52. */
int bis_spmv_jacobi(bis_context *ctx, const bis_matrix *A, const double *D,
                    const double *b, const double *x_old, double *x_new);
/* The same sweep fused with the residual of the iterate it starts from: r = b - A x_old (stored if r != NULL),
 * slot_rr <- (r,r), x_new as above -- one product A x_old serves jacobi.hpp:27-52 and the residual sampling of
 * jacobi.hpp:102-107 that the reference's harness does with a second SpMV. */
int bis_spmv_jacobi_residual(bis_context *ctx, const bis_matrix *A, const double *D, const double *b,
                             const double *x_old, double *x_new, double *r, int slot_rr);
/* out = b - T x for a strictly triangular T: gauss_seidel.hpp:30-34, 44-48. */
int bis_spmv_sub(bis_context *ctx, const bis_matrix *T, const double *x,
                 const double *b, double *out);
/* One inner iteration of two_stage_gauss_seidel (kernels.hpp:321-331), fused:
 * work_out = (D_inv * -1) * (T work_in) ; output = output + work_out. */
int bis_spmv_two_stage(bis_context *ctx, const bis_matrix *T, const double *D_inv /* [dev] */,
                       const double *work_in /* [dev] */, double *work_out /* [dev] */,
                       double *output /* [dev] */);

/* CG, methods/cg.hpp:6-54.
 * alpha = s[rz]/s[pAp]; x_new = x_old + alpha p_old; r_new = r_old - alpha Ap;
 * s[rr] <- (r_new,r_new); precond NONE: z_new = r_new; JACOBI: z_new =
 * r_new / A_D; both: s[rz_new] <- (r_new,z_new).  Other preconditioners:
 * z_new untouched, s[rz_new] untouched (caller applies M^-1 then
 * bis_dot_to_slot).  x_new == NULL: no x update (see bis_cg_direction_x). */
int bis_cg_update(bis_context *ctx, int precond, int64_t n, double *x_new,
                  const double *x_old, const double *p_old, double *r_new,
                  const double *r_old, const double *Ap, double *z_new,
                  const double *A_D, int slot_rz, int slot_pAp, int slot_rr,
                  int slot_rz_new);
/* beta = s[rz_new]/s[rz]; p_new = z_new + beta p_old (cg.hpp:47-52) */
int bis_cg_direction(bis_context *ctx, int64_t n, double *p_new,
                     const double *z_new, const double *p_old, int slot_rz_new,
                     int slot_rz);
/* The same plus the x update of cg.hpp:27-28 (x_new = x_old + alpha p_old,
 * alpha = s[rz]/s[pAp]) in one pass over p_old; pair it with bis_cg_update
 * called with x_new == NULL, which then skips the x update. */
int bis_cg_direction_x(bis_context *ctx, int64_t n, double *p_new,
                       const double *z_new, const double *p_old, double *x_new,
                       const double *x_old, int slot_rz_new, int slot_rz,
                       int slot_pAp);

/* BiCGSTAB, methods/bicgstab.hpp:8-83.
 * alpha = s[rho_old]/s[r0v]; s = r_old - alpha v; JACOBI: s_tmp = s / A_D,
 * NONE: s_tmp = s (copy); other: s_tmp untouched. */
int bis_bicgstab_s(bis_context *ctx, int precond, int64_t n, double *s,
                   double *s_tmp, const double *r_old, const double *v,
                   const double *A_D, int slot_rho_old, int slot_r0v);
/* alpha as above; omega = s[zs]/s[zz]; h = x_old + alpha y (stored if
 * h != NULL); x_new = h + omega s_tmp; r_new = s - omega z;
 * s[rho_new] <- (r0,r_new); s[rr] <- (r_new,r_new).  bicgstab.hpp:51-68. */
int bis_bicgstab_xr(bis_context *ctx, int64_t n, double *h, double *x_new,
                    const double *x_old, const double *y, const double *s_tmp,
                    double *r_new, const double *s, const double *z,
                    const double *r0, int slot_rho_old, int slot_r0v,
                    int slot_zs, int slot_zz, int slot_rho_new, int slot_rr);
/* beta = (s[rho_new]/s[rho_old])*(alpha/omega); tmp = p_old - omega v (stored
 * if tmp != NULL); p_new = r_new + beta tmp; y_next = M^-1 p_new for NONE
 * (copy) / JACOBI (divide) when y_next != NULL.  bicgstab.hpp:70-78 and the
 * next iteration's :24-27. */
int bis_bicgstab_p(bis_context *ctx, int precond, int64_t n, double *tmp,
                   double *p_new, const double *p_old, const double *v,
                   const double *r_new, double *y_next, const double *A_D,
                   int slot_rho_new, int slot_rho_old, int slot_r0v,
                   int slot_zs, int slot_zz);

/* GMRES, methods/gmres.hpp.
 * Modified Gram-Schmidt step j (gmres.hpp:6-53): w -= s[h_j] v_j, then
 * s[out] <- (w, v_next), or (w,w) when v_next == NULL.  The arithmetic is
 * the reference's dot -> axpy -> dot chain; only the passes are merged. */
int bis_mgs_step(bis_context *ctx, int64_t n, double *w, const double *v_j,
                 const double *v_next, int slot_h_j, int slot_out);
/* out = w * (1.0 / sqrt(s[sumsq])) (gmres.hpp:36-45, :305) */
int bis_scale_inv_norm(bis_context *ctx, int64_t n, double *out,
                       const double *w, int slot_sumsq);
/* get_explicit_x (gmres.hpp:326-375): Vy = sum_{j<k} V_j y[j] ; x = x_old +
 * Vy.  V is (m+1) x n row-major [dev], y [host] has k entries (F6: the
 * reference's out-of-bounds y[k] term is defined as 0). */
int bis_gmres_update_x(bis_context *ctx, int64_t n, int k, const double *V,
                       const double *y /* [host] */, double *x,
                       const double *x_old, double *Vy);

/* ---- multiple right-hand sides -----------------------------------------
 * New in the build: the reference solves one right-hand side at a time.
 * Several systems with the same matrix (load cases, sources, sweeps over b)
 * share ONE pass over the matrix per iteration.  Single-GPU contexts only.
 *
 * Layout: a block of k vectors (1 <= k <= BIS_BLOCK_MAX_K) is an n x k
 * ROW-MAJOR device array, element (i, j) at V[i*k + j], allocated with
 * bis_vector_alloc(ctx, n*k) (16-byte aligned; every block argument must be).
 * A numpy / torch (n, k) C-contiguous array uploads as is.  Column j's
 * scalars live in slots slot0 + j; slot0 + k > BIS_NUM_SCALARS is an error.
 *
 * Every column is bit-identical to the single-vector entry point it batches:
 * bis_spmm to native_spmv (products rounded separately, added in storage
 * order; = bis_spmv wherever that takes the TMA-tile or windowed variant),
 * the streaming kernels to bis_dot_to_slot / bis_subtract_vectors /
 * bis_elemwise_div_vectors / bis_cg_update / bis_cg_direction_x (same rows
 * per block, same accumulation order, same reduction tree).  All are
 * enqueue-only (graph-recordable).  They fail on a distributed context, k
 * outside [1, 16], a block argument that is not 16-byte aligned and a matrix
 * without CRS arrays (option factor_keep_crs = 0).
 *
 * `state` [dev] of a block CG: 3k doubles, [0,k) stop thresholds
 * tol*||r0_j||, [k,2k) active flags (1.0 / 0.0), [2k,3k) iterations done;
 * NULL = every column active.  A column that is not active is frozen: its
 * vectors and slots are not written, except that the direction step carries
 * its x through (X_new = X_old), so the final iterate of every column is
 * always in the X_new of the last step. */
#define BIS_BLOCK_MAX_K 16
/* Y = A X, X: n_cols x k, Y: n_rows x k.  Counted in the "spmv" profile
 * family, NVTX range "spmm". */
int bis_spmm(bis_context *ctx, const bis_matrix *A, int k, const double *X /* [dev] */,
             double *Y /* [dev] */);
/* slot0 + j <- (A_j, B_j) for every column j (active ones only if state). */
int bis_block_dot_to_slots(bis_context *ctx, int64_t n, int k, const double *A,
                           const double *B, int slot0, const double *state);
/* Initial residual of a block CG (cg.hpp:100-120 per column): R = B - AX,
 * Z = M^-1 R (precond NONE: copy, JACOBI: R / A_D), P = Z if P != NULL,
 * slot_rz0 + j <- (r_j, z_j), slot_rr0 + j <- (r_j, r_j). */
int bis_block_residual(bis_context *ctx, int precond, int64_t n, int k,
                       const double *AX, const double *B, const double *A_D,
                       double *R, double *Z, double *P, int slot_rz0,
                       int slot_rr0);
/* bis_cg_update (x_new = NULL) per column: alpha_j = s[rz0+j]/s[pAp0+j];
 * R_new = R_old - alpha AP; Z_new = R_new or R_new / A_D; s[rr0+j] <-
 * (r,r); s[rz_new0+j] <- (r,z).  Precond NONE or JACOBI only. */
int bis_block_cg_update(bis_context *ctx, int precond, int64_t n, int k,
                        double *R_new, const double *R_old, const double *AP,
                        double *Z_new, const double *A_D, int slot_rz0,
                        int slot_pAp0, int slot_rr0, int slot_rz_new0,
                        const double *state);
/* bis_cg_direction_x per column: X_new = X_old + alpha P_old, P_new = Z_new
 * + beta P_old (inactive columns: X_new = X_old, P_new untouched). */
int bis_block_cg_direction_x(bis_context *ctx, int64_t n, int k, double *P_new,
                             const double *Z_new, const double *P_old,
                             double *X_new, const double *X_old,
                             int slot_rz_new0, int slot_rz0, int slot_pAp0,
                             const double *state);
/* Start of a block-CG iteration: the stop rule of the harness
 * (solver.hpp:173-191) on the device, latched for the whole iteration.  An
 * active column that has run >= 1 iteration stops when sqrt(s[rr0+j]) <
 * threshold, > DBL_MAX or NaN; one that has run max_iters stops; every
 * column still active counts the iteration. */
int bis_block_cg_status(bis_context *ctx, int k, int slot_rr0, int max_iters,
                        double *state /* [dev] */);

#ifdef __cplusplus
}
#endif
#endif /* BIS_B200_H */
