// host/methods/block_cg.hpp -- CG on k right-hand sides with the same matrix (new in the build; the reference
// solves one b at a time).  Every column runs exactly the iteration of ConjugateGradientSolver (methods/cg.hpp)
// with preconditioner none or jacobi; the columns share one pass over the matrix per iteration (bis_spmm):
//   status: latch which columns are still active               bis_block_cg_status
//   AP = A P_old ; (AP_j, p_j)                                 bis_spmm + bis_block_dot_to_slots
//   alpha ; R_new ; (r,r) ; Z_new ; (r,z)                      bis_block_cg_update
//   beta ; P_new ; X_new = X_old + alpha P_old                 bis_block_cg_direction_x
// A column stops by the harness's rule (solver.hpp: check_stopping_criteria), decided on the device from its own
// residual, so the iteration body stays enqueue-only (recorded as a CUDA graph, period 2) and the host runs one
// iteration ahead of the residual read-back, as the single-RHS CG does.  The host replays the same decisions from
// the same numbers to keep the per-column histories.  Stopped columns are frozen; their x is carried through
// (X_new = X_old), so X_old after the last exchange holds the final iterate of every column.
#pragma once

#include "../solver.hpp"

// slots: [S_B_RR, +k) (r,r) of the newest residual; two banks of (r,z) swapped like the vectors; (Ap,p)
enum BlockSlot : int { S_B_RR = 32, S_B_RZ_A = 48, S_B_RZ_B = 64, S_B_PAP = 80 };

// What the block solvers whose iteration starts with bis_block_cg_status and ends with the k (r,r) slots at S_B_RR share
// (block CG, block Gauss-Seidel): the device state, the host mirror of the per-column stop decisions, and the loop.
class BlockSolver : public Solver {
  public:
    int k = 0;
    double *state = nullptr;   // [3k] device stop state (bis_block_cg_status)
    std::vector<double> threshold;
    std::vector<int> col_iters;
    std::vector<char> col_active, col_converged;
    std::vector<std::vector<double>> col_history;

    BlockSolver(const Args *cli_args, Interface *device, int k_) : Solver(cli_args, device), k(k_) {}

    // rr: (r_j, r_j) of the initial residuals; state must be allocated
    void init_columns(const double *rr) {
        threshold.assign(k, 0.0);
        col_iters.assign(k, 0);
        col_active.assign(k, 1);
        col_converged.assign(k, 0);
        col_history.assign(k, {});
        std::vector<double> st(3 * k, 0.0);
        for (int j = 0; j < k; ++j) {
            const double r0 = std::sqrt(rr[j]);
            col_history[j].push_back(r0);
            threshold[j] = tolerance * r0;   // init_stopping_criteria
            st[j] = threshold[j];
            st[k + j] = 1.0;
        }
        BIS_OK(bis_vector_upload(dev, state, st.data(), 3 * k));
    }
    int n_active() const {
        int a = 0;
        for (char c : col_active) a += c ? 1 : 0;
        return a;
    }
    // the residuals of iteration `iter`, read back: history and stop decision of every column active in it
    void record(const double *rr, int iter) {
        for (int j = 0; j < k; ++j) {
            if (!col_active[j]) continue;
            const double nrm = std::sqrt(rr[j]);
            col_history[j].push_back(nrm);
            col_iters[j] = iter;
            const bool conv = std::abs(nrm) < threshold[j];
            if (conv || iter >= max_iters || std::abs(nrm) > DBL_MAX || std::isnan(nrm)) {
                col_active[j] = 0;
                col_converged[j] = conv ? 1 : 0;
            }
        }
    }
    // The loop: one read-back of the k (r,r) slots per iteration, the next iteration enqueued before waiting
    // for it.  timer_from > 0: device events around iterations timer_from+1 .. the last (measurements).
    void run(int timer_from = 0, double *timed_ms = nullptr, int *timed_iters = nullptr) {
        std::vector<double> rr(k);
        bool ahead = false;
        bool timing = false;
        int first_timed = 0;
        while (n_active() > 0) {
            if (!ahead) {
                if (timer_from > 0 && iter_count == timer_from && !timing) {
                    BIS_OK(bis_timer_start(dev));
                    timing = true;
                    first_timed = iter_count;
                }
                iterate(nullptr);
            }
            ahead = false;
            ++iter_count;
            BIS_OK(bis_scalar_read_begin(dev, S_B_RR, k));
            exchange();
            if (iter_count < max_iters) {
                if (timer_from > 0 && iter_count == timer_from && !timing) {
                    BIS_OK(bis_timer_start(dev));
                    timing = true;
                    first_timed = iter_count;
                }
                iterate(nullptr);
                ahead = true;
            }
            BIS_OK(bis_scalar_read_end(dev, S_B_RR, k, rr.data()));
            record(rr.data(), iter_count);
        }
        if (timing) {
            double ms = 0.0;
            BIS_OK(bis_timer_stop(dev, &ms));   // also covers a last iteration run ahead
            if (timed_ms) *timed_ms = ms;
            if (timed_iters) *timed_iters = iter_count + (ahead ? 1 : 0) - first_timed;
        }
        BIS_OK(bis_context_synchronize(dev));
    }
};

class BlockCGSolver : public BlockSolver {
  public:
    double *X_new = nullptr, *X_old = nullptr, *P_new = nullptr, *P_old = nullptr;
    double *R_new = nullptr, *R_old = nullptr, *Z_new = nullptr, *Z_old = nullptr;
    double *AP = nullptr, *B = nullptr, *D = nullptr;
    int s_rz = S_B_RZ_A, s_rz_new = S_B_RZ_B;

    BlockCGSolver(const Args *cli_args, Interface *device, int k_) : BlockSolver(cli_args, device, k_) {
        if (k < 1 || k > BIS_BLOCK_MAX_K) bis_fatal("block CG: k outside [1, BIS_BLOCK_MAX_K]");
        if (preconditioner != PrecondType::None && preconditioner != PrecondType::Jacobi)
            bis_fatal("block CG: preconditioner " + to_string(preconditioner) + " not supported (none or jacobi)");
    }

    // n rows; B_host / X0_host: n x k row-major host arrays (X0 NULL: INIT_X_VAL everywhere)
    void setup(std::unique_ptr<DeviceCRS> A, const double *B_host, const double *X0_host) {
        dA = std::move(A);
        N = dA->n_rows;
        N_global = dA->n_rows_global;
        const int64_t nk = N * k;
        for (double **p : {&X_new, &X_old, &P_new, &P_old, &R_new, &R_old, &Z_new, &Z_old, &AP, &B}) *p = dev_new(dev, nk);
        state = dev_new(dev, 3 * k);
        BIS_OK(bis_vector_upload(dev, B, B_host, nk));
        if (X0_host) BIS_OK(bis_vector_upload(dev, X_old, X0_host, nk));
        else init_vector(dev, X_old, INIT_X_VAL, nk);
        init_vector(dev, X_new, 0.0, nk);
        if (preconditioner == PrecondType::Jacobi) {
            D = dev_new(dev, N);
            BIS_OK(bis_matrix_extract_diagonal(dev, dA->handle, D, nullptr));
        }
        // cg.hpp:100-120 per column: R = B - A X0, Z = M^-1 R, P = Z, (r,z), (r,r)
        BIS_OK(bis_spmm(dev, dA->handle, k, X_old, AP));
        BIS_OK(bis_block_residual(dev, static_cast<int>(preconditioner), N, k, AP, B, D, R_old, Z_old, P_old, s_rz, S_B_RR));
        std::vector<double> rr(k);
        BIS_OK(bis_scalar_get(dev, S_B_RR, k, rr.data()));
        init_columns(rr.data());
    }

    void iterate(Timers *) override {
        graphed(exchange_count & 1, [&] {
            const int pc = static_cast<int>(preconditioner);
            BIS_OK(bis_block_cg_status(dev, k, S_B_RR, max_iters, state));
            BIS_OK(bis_spmm(dev, dA->handle, k, P_old, AP));
            BIS_OK(bis_block_dot_to_slots(dev, N, k, AP, P_old, S_B_PAP, state));
            BIS_OK(bis_block_cg_update(dev, pc, N, k, R_new, R_old, AP, Z_new, D, s_rz, S_B_PAP, S_B_RR, s_rz_new, state));
            BIS_OK(bis_block_cg_direction_x(dev, N, k, P_new, Z_new, P_old, X_new, X_old, s_rz_new, s_rz, S_B_PAP, state));
        });
    }
    void exchange() override {
        ++exchange_count;
        std::swap(P_old, P_new);
        std::swap(Z_old, Z_new);
        std::swap(R_old, R_new);
        std::swap(X_old, X_new);
        std::swap(s_rz, s_rz_new);
    }
    // ||b_j - A x*_j|| of every column (x* = X_old); R_new / Z_new are scratch here
    std::vector<double> true_residuals() {
        BIS_OK(bis_spmm(dev, dA->handle, k, X_old, AP));
        BIS_OK(bis_block_residual(dev, BIS_PRECOND_NONE, N, k, AP, B, nullptr, R_new, Z_new, nullptr, S_B_PAP, S_B_RR));
        std::vector<double> rr(k);
        BIS_OK(bis_scalar_get(dev, S_B_RR, k, rr.data()));
        for (double &v : rr) v = std::sqrt(v);
        return rr;
    }
    ~BlockCGSolver() override {
        for (double **p : {&X_new, &X_old, &P_new, &P_old, &R_new, &R_old, &Z_new, &Z_old, &AP, &B, &D, &state})
            dev_delete(dev, *p);
    }
};
