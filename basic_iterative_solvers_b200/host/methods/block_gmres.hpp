// host/methods/block_gmres.hpp -- restarted GMRES on k right-hand sides with the same matrix (new in the build; the
// reference solves one b at a time).  Column j runs exactly the arithmetic of GMRESSolver (methods/gmres.hpp) on b_j
// with preconditioner none or jacobi: the same stop rule, restarts and history.  The device part of an iteration at
// basis index i is i + 4 launches, recorded as a CUDA graph keyed by i:
//   W = A V_i                                                bis_spmm
//   W = M^-1 W ; h_0 = (W, V_0)                              bis_block_gmres_precond_dot
//   W -= h_l V_l ; h_{l+1} = (W, V_{l+1}), or (W, W) at l=i  bis_block_mgs_step, l = 0..i
//   V_{i+1} = W / ||W||                                      bis_block_scale_inv_norm
// One split read fetches the Hessenberg column of every column; the next body is enqueued behind it (under the
// single-RHS condition) while the host runs each column's Givens update (least_squares / update_g of gmres.hpp).
// A column stops by check_stopping_criteria; its x is formed then (get_explicit_x: back-substitution, masked
// bis_block_gmres_update_x) and its active flag on the device is cleared, which freezes it in every later kernel.
// Columns still running restart together, so they share one restart count.
#pragma once

#include "gmres.hpp"

#include <chrono>

// slots of the (r,z) / (r,r) reductions of bis_block_residual
enum BlockGMRESSlot : int { S_BG_RZ = 32, S_BG_RR = 48 };

class BlockGMRESSolver : public Solver {
  public:
    int k = 0, m = 0;
    int64_t ldv = 0;   // basis stride: n*k rounded up to even, so every V_l is 16-byte aligned
    // X holds x and x_old of every column at once: get_explicit_x is x = x_old + V y with x_old == x (gmres.hpp
    // keeps them equal outside that step), so the update runs in place.
    double *X = nullptr, *B = nullptr, *W = nullptr, *R = nullptr, *Z = nullptr;   // n x k [dev]
    double *V = nullptr, *H = nullptr, *D = nullptr, *active = nullptr;            // [dev]
    struct Column {   // GMRESSolver's host state, one per right-hand side
        std::vector<double> y, H, H_tmp, J, Q, Q_tmp, R, g, g_tmp, history;
        double beta = 0.0, threshold = 0.0, residual_norm = 0.0;
        int iters = 0, restarts = 0;
        bool active = true, converged = false;
    };
    std::vector<Column> col;
    double givens_s = 0.0;   // host seconds in least_squares / update_g, all columns and iterations

    BlockGMRESSolver(const Args *cli_args, Interface *device, int k_) : Solver(cli_args, device), k(k_) {
        m = gmres_restart_len;
        if (k < 1 || k > BIS_BLOCK_MAX_K) bis_fatal("block GMRES: k outside [1, BIS_BLOCK_MAX_K]");
        if (m < 1 || m > BIS_BLOCK_GMRES_MAX_M) bis_fatal("GMRES restart length must be in [1, 64]");
        if (preconditioner != PrecondType::None && preconditioner != PrecondType::Jacobi)
            bis_fatal("block GMRES: preconditioner " + to_string(preconditioner) + " not supported (none or jacobi)");
    }

    // n rows; B_host / X0_host: n x k row-major host arrays (X0 NULL: INIT_X_VAL everywhere)
    void setup(std::unique_ptr<DeviceCRS> A, const double *B_host, const double *X0_host) {
        dA = std::move(A);
        N = dA->n_rows;
        N_global = dA->n_rows_global;
        const int64_t nk = N * k;
        ldv = (nk + 1) & ~(int64_t)1;
        for (double **p : {&X, &B, &W, &R, &Z}) *p = dev_new(dev, nk);
        V = dev_new(dev, ldv * (m + 1));
        H = dev_new(dev, (int64_t)(m + 2) * k);
        active = dev_new(dev, k);
        BIS_OK(bis_vector_upload(dev, B, B_host, nk));
        if (X0_host) BIS_OK(bis_vector_upload(dev, X, X0_host, nk));
        else init_vector(dev, X, INIT_X_VAL, nk);
        if (preconditioner == PrecondType::Jacobi) {
            D = dev_new(dev, N);
            BIS_OK(bis_matrix_extract_diagonal(dev, dA->handle, D, nullptr));
        }
        col.assign(k, Column{});
        for (Column &c : col) {
            c.y.assign(m + 1, 0.0);
            for (auto *v : {&c.H, &c.H_tmp, &c.R}) v->assign((size_t)(m + 1) * m, 0.0);
            for (auto *v : {&c.J, &c.Q, &c.Q_tmp}) v->assign((size_t)(m + 1) * (m + 1), 0.0);
            c.g.assign(m + 1, 0.0);
            c.g_tmp.assign(m + 1, 0.0);
        }
        upload_active();
        init_residual_block(true);
    }

    void upload_active() {
        std::vector<double> f(k);
        for (int j = 0; j < k; ++j) f[j] = col[j].active ? 1.0 : 0.0;
        BIS_OK(bis_vector_upload(dev, active, f.data(), k));
    }

    // init_structs + init_residual (gmres.hpp) for every active column: R = B - A X, Z = M^-1 R, beta^2 = (z,z),
    // V_0 = Z / beta.  V_1..V_m are not zeroed as init_structs does: each is written before it is read.
    void init_residual_block(bool first) {
        BIS_OK(bis_spmm(dev, dA->handle, k, X, W));
        BIS_OK(bis_block_residual(dev, static_cast<int>(preconditioner), N, k, W, B, D, R, Z, nullptr, S_BG_RZ, S_BG_RR));
        BIS_OK(bis_block_gmres_precond_dot(dev, BIS_PRECOND_NONE, N, k, Z, nullptr, nullptr, H, active));
        BIS_OK(bis_block_scale_inv_norm(dev, N, k, V, Z, H, 0, active));
        std::vector<double> beta2(k), rr(k);
        BIS_OK(bis_vector_read_begin(dev, H, k));
        BIS_OK(bis_vector_read_end(dev, beta2.data(), k));
        if (first) BIS_OK(bis_scalar_get(dev, S_BG_RR, k, rr.data()));
        for (int j = 0; j < k; ++j) {
            Column &c = col[j];
            if (!c.active) continue;
            if (first) {
                c.residual_norm = std::sqrt(rr[j]);   // the unpreconditioned ||r0||
                c.history.push_back(c.residual_norm);
                c.threshold = tolerance * c.residual_norm;   // init_stopping_criteria
            }
            std::fill(c.y.begin(), c.y.end(), 0.0);
            for (auto *v : {&c.g, &c.g_tmp, &c.H, &c.H_tmp, &c.R}) std::fill(v->begin(), v->end(), 0.0);
            init_dense_identity_matrix(c.J.data(), m + 1, m + 1);
            init_dense_identity_matrix(c.Q.data(), m + 1, m + 1);
            init_dense_identity_matrix(c.Q_tmp.data(), m + 1, m + 1);
            c.beta = std::sqrt(beta2[j]);
            c.g[0] = c.beta;
            c.g_tmp[0] = c.beta;
            if (!first) {
                c.residual_norm = c.beta;
                c.history.push_back(c.beta);
            }
        }
    }

    void enqueue_iteration(const int i) {
        graphed(i, [&] {
            const int pc = static_cast<int>(preconditioner);
            BIS_OK(bis_spmm(dev, dA->handle, k, V + i * ldv, W));
            BIS_OK(bis_block_gmres_precond_dot(dev, pc, N, k, W, D, V, H, active));
            for (int l = 0; l <= i; ++l)
                BIS_OK(bis_block_mgs_step(dev, N, k, W, V + l * ldv, l < i ? V + (l + 1) * ldv : nullptr, H, l, active));
            BIS_OK(bis_block_scale_inv_norm(dev, N, k, V + (i + 1) * ldv, W, H, i + 1, active));
        });
    }
    void iterate(Timers *) override { enqueue_iteration(iter_count - gmres_restart_count * m); }
    void exchange() override {}

    int n_active() const {
        int a = 0;
        for (const Column &c : col) a += c.active ? 1 : 0;
        return a;
    }
    bool stops(const Column &c) const {   // check_stopping_criteria (solver.hpp)
        const double r = c.residual_norm;
        return std::abs(r) < c.threshold || iter_count >= max_iters - c.restarts || std::abs(r) > DBL_MAX || std::isnan(r);
    }
    // get_explicit_x of the columns in `mask` over the first nb basis blocks
    void explicit_x(const std::vector<int> &mask, int nb) {
        std::vector<double> Y((size_t)k * nb, 0.0);
        for (int j = 0; j < k; ++j) {
            if (!mask[j]) continue;
            Column &c = col[j];
            back_substitution(nb, m, c.R.data(), c.g.data(), c.y.data());
            for (int l = 0; l < nb; ++l) Y[(size_t)j * nb + l] = c.y[l];
        }
        BIS_OK(bis_block_gmres_update_x(dev, N, k, nb, V, ldv, Y.data(), X, X, mask.data()));
    }
    // the columns in `mask` stop here: final x, frozen from now on
    void finish(const std::vector<int> &mask, int nb) {
        bool any = false;
        for (int j = 0; j < k; ++j) any = any || mask[j];
        if (!any) return;
        explicit_x(mask, nb);
        for (int j = 0; j < k; ++j)
            if (mask[j]) {
                col[j].active = false;
                col[j].converged = col[j].residual_norm < col[j].threshold;
            }
        upload_active();
    }

    // The loop of solve() (solver_harness.hpp) for all columns at once.  timer_from > 0: device events around
    // iterations timer_from+1 .. the last (measurements).
    void run(int timer_from = 0, double *timed_ms = nullptr, int *timed_iters = nullptr) {
        std::vector<double> hcol((size_t)(m + 2) * k);
        bool ahead = false, timing = false;
        int first_timed = 0;
        auto enqueue = [&](int i, int iteration) {
            if (timer_from > 0 && iteration == timer_from && !timing) {
                BIS_OK(bis_timer_start(dev));
                timing = true;
                first_timed = iteration;
            }
            enqueue_iteration(i);
        };
        while (n_active() > 0) {
            const int i = iter_count - gmres_restart_count * m;
            if (!ahead) enqueue(i, iter_count);
            ahead = false;
            BIS_OK(bis_vector_read_begin(dev, H, (int64_t)(i + 2) * k));
            if (i + 1 < m && iter_count + 1 < max_iters - gmres_restart_count) {
                enqueue(i + 1, iter_count + 1);
                ahead = true;
            }
            BIS_OK(bis_vector_read_end(dev, hcol.data(), (int64_t)(i + 2) * k));
            const auto t0 = std::chrono::steady_clock::now();
            for (int j = 0; j < k; ++j) {   // GMRESSolver::iterate's host part
                Column &c = col[j];
                if (!c.active) continue;
                for (int l = 0; l <= i; ++l) c.H[i + l * m] = hcol[(size_t)l * k + j];
                c.H[(i + 1) * m + i] = std::sqrt(hcol[(size_t)(i + 1) * k + j]);
                least_squares(i, m, c.J.data(), c.H.data(), c.H_tmp.data(), c.Q.data(), c.Q_tmp.data(), c.R.data());
                update_g(i, m, c.Q.data(), c.g.data(), c.g_tmp.data(), c.residual_norm, c.beta);
            }
            givens_s += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            ++iter_count;
            // sample_residual, then check_restart (gmres.hpp:388-415), then check_stopping_criteria, per column
            const bool cycle = iter_count % m == 0;
            std::vector<int> restart(k, 0), stop(k, 0);
            bool any_restart = false;
            for (int j = 0; j < k; ++j) {
                Column &c = col[j];
                if (!c.active) continue;
                c.history.push_back(c.residual_norm);
                c.iters = iter_count;
                restart[j] = !(c.residual_norm < c.threshold) && !(iter_count > max_iters) && cycle;
                any_restart = any_restart || restart[j];
                if (!restart[j]) stop[j] = stops(c);
            }
            finish(stop, i + 1);
            if (any_restart) {
                explicit_x(restart, i + 1);
                init_residual_block(false);
                ++gmres_restart_count;
                for (int j = 0; j < k; ++j) {
                    if (!restart[j]) continue;
                    col[j].restarts = gmres_restart_count;
                    stop[j] = stops(col[j]);
                }
                finish(stop, 0);   // a column that stops right after its restart: x = x_old + 0 (get_explicit_x, k = 0)
            }
        }
        if (timing) {
            double ms = 0.0;
            BIS_OK(bis_timer_stop(dev, &ms));   // also covers a last iteration run ahead
            if (timed_ms) *timed_ms = ms;
            if (timed_iters) *timed_iters = iter_count + (ahead ? 1 : 0) - first_timed;
        }
        BIS_OK(bis_context_synchronize(dev));
    }
    // ||b_j - A x*_j|| of every column; W, R, Z are scratch here
    std::vector<double> true_residuals() {
        BIS_OK(bis_spmm(dev, dA->handle, k, X, W));
        BIS_OK(bis_block_residual(dev, BIS_PRECOND_NONE, N, k, W, B, nullptr, R, Z, nullptr, S_BG_RZ, S_BG_RR));
        std::vector<double> rr(k);
        BIS_OK(bis_scalar_get(dev, S_BG_RR, k, rr.data()));
        for (double &v : rr) v = std::sqrt(v);
        return rr;
    }
    ~BlockGMRESSolver() override {
        for (double **p : {&X, &B, &W, &R, &Z, &V, &H, &D, &active}) dev_delete(dev, *p);
    }
};
