// host/methods/block_gs.hpp -- Gauss-Seidel and symmetric Gauss-Seidel on k right-hand sides with the same matrix
// (new in the build; the reference solves one b at a time).  Column j runs exactly GaussSeidelSolver /
// SymmetricGaussSeidelSolver (methods/gauss_seidel.hpp) on b_j; the columns share one pass over each factor per sweep,
// and the triangular solves carry all k values through each dependency of the level schedule:
//   status: latch which columns are still active          bis_block_cg_status
//   T = B - U X ; X = (D+L)^-1 T                           bis_spmm_sub + bis_block_sptrsv
//   SGS only:  T = B - L X ; X = (D+U)^-1 T                bis_spmm_sub + bis_block_bsptrsv
//   AX = A X ; R = B - AX, (r,r)                           bis_spmm + bis_block_residual
// X is updated in place, as in the single-RHS solver.  The triangular solves skip the columns that have stopped, so a
// column keeps the iterate it stopped on even when the host has run one iteration ahead.  Stop rule, graph and
// run-ahead are those of block CG (BlockSolver).
#pragma once

#include "block_cg.hpp"

class BlockGSSolver : public BlockSolver {
  public:
    bool symmetric = false;
    double *X = nullptr, *T = nullptr, *AX = nullptr, *R = nullptr, *Z = nullptr, *B = nullptr, *D = nullptr;

    BlockGSSolver(const Args *cli_args, Interface *device, int k_, bool sgs)
        : BlockSolver(cli_args, device, k_), symmetric(sgs) {
        const std::string name = sgs ? "block SGS" : "block GS";
        if (k < 1 || k > BIS_BLOCK_MAX_K) bis_fatal(name + ": k outside [1, BIS_BLOCK_MAX_K]");
        if (preconditioner != PrecondType::None)
            bis_fatal(name + ": preconditioner " + to_string(preconditioner) + " not supported (the stationary methods take none)");
    }

    // n rows; B_host / X0_host: n x k row-major host arrays (X0 NULL: INIT_X_VAL everywhere)
    void setup(std::unique_ptr<DeviceCRS> A, const double *B_host, const double *X0_host) {
        dA = std::move(A);
        N = dA->n_rows;
        N_global = dA->n_rows_global;
        const int64_t nk = N * k;
        for (double **p : {&X, &T, &AX, &R, &Z, &B}) *p = dev_new(dev, nk);
        state = dev_new(dev, 3 * k);
        D = dev_new(dev, N);
        BIS_OK(bis_vector_upload(dev, B, B_host, nk));
        if (X0_host) BIS_OK(bis_vector_upload(dev, X, X0_host, nk));
        else init_vector(dev, X, INIT_X_VAL, nk);
        BIS_OK(bis_matrix_extract_diagonal(dev, dA->handle, D, nullptr));
        // the sweeps multiply by the factors: they keep their natural-order CRS whatever the context option says
        int keep_before = 1;
        BIS_OK(bis_context_get_option(dev, "factor_keep_crs", &keep_before));
        struct RestoreOption {
            Interface *dev;
            int value;
            ~RestoreOption() { bis_context_set_option(dev, "factor_keep_crs", value); }
        } restore_keep{dev, keep_before};
        BIS_OK(bis_context_set_option(dev, "factor_keep_crs", 1));
        bis_matrix *l = nullptr, *u = nullptr;
        BIS_OK(bis_matrix_split_triangular(dev, dA->handle, &l, &u));
        dL_strict = adopt_device_matrix(dev, l);
        dU_strict = adopt_device_matrix(dev, u);
        BIS_OK(bis_spmm(dev, dA->handle, k, X, AX));
        BIS_OK(bis_block_residual(dev, BIS_PRECOND_NONE, N, k, AX, B, nullptr, R, Z, nullptr, S_B_RZ_A, S_B_RR));
        std::vector<double> rr(k);
        BIS_OK(bis_scalar_get(dev, S_B_RR, k, rr.data()));
        init_columns(rr.data());
    }

    void iterate(Timers *) override {
        graphed(0, [&] {
            const double *active = state + k;
            BIS_OK(bis_block_cg_status(dev, k, S_B_RR, max_iters, state));
            BIS_OK(bis_spmm_sub(dev, dU_strict->handle, k, X, B, T));               // T <- B - U X
            BIS_OK(bis_block_sptrsv(dev, dL_strict->handle, k, X, D, T, active));   // X <- (D+L)^-1 T
            if (symmetric) {
                BIS_OK(bis_spmm_sub(dev, dL_strict->handle, k, X, B, T));            // T <- B - L X
                BIS_OK(bis_block_bsptrsv(dev, dU_strict->handle, k, X, D, T, active));   // X <- (D+U)^-1 T
            }
            BIS_OK(bis_spmm(dev, dA->handle, k, X, AX));
            BIS_OK(bis_block_residual(dev, BIS_PRECOND_NONE, N, k, AX, B, nullptr, R, Z, nullptr, S_B_RZ_A, S_B_RR));
        });
    }
    void exchange() override { ++exchange_count; }
    // ||b_j - A x*_j|| of every column (x* = X); R / Z are scratch here
    std::vector<double> true_residuals() {
        BIS_OK(bis_spmm(dev, dA->handle, k, X, AX));
        BIS_OK(bis_block_residual(dev, BIS_PRECOND_NONE, N, k, AX, B, nullptr, R, Z, nullptr, S_B_PAP, S_B_RR));
        std::vector<double> rr(k);
        BIS_OK(bis_scalar_get(dev, S_B_RR, k, rr.data()));
        for (double &v : rr) v = std::sqrt(v);
        return rr;
    }
    ~BlockGSSolver() override {
        for (double **p : {&X, &T, &AX, &R, &Z, &B, &D, &state}) dev_delete(dev, *p);
    }
};
