// host/methods/gmres.hpp -- restarted GMRES (reference methods/gmres.hpp).
// Device side: w = A V[k], M^-1 w, modified Gram-Schmidt (gmres.hpp:6-53) as
// fused axpy+dot launches (the reference's dot -> axpy -> dot chain, one pass
// over w per basis vector instead of two), the basis normalisation and
// get_explicit_x's N x k product.  Host side, restated literally: the Givens
// least-squares update on the (m+1) x m Hessenberg matrix (gmres.hpp:55-148) and
// the k x k back-substitution (gmres.hpp:335-349).  One host<->device sync per
// iteration fetches the new Hessenberg column; the next iteration's device work is
// already enqueued behind it.
//
// SURVEY.md F6: the reference's get_explicit_x reads y[k] one past the end of
// `y` when k == m; the term is defined here as 0 (sum over j < k).
#pragma once

#include "../solver.hpp"

// gmres.hpp:55-121
inline void least_squares(int n_solver_iters, int restart_len, double *J, double *H, double *H_tmp,
                          double *Q, double *Q_tmp, double *R) {
    const int m = restart_len, k = n_solver_iters;
    init_dense_identity_matrix(J, m + 1, m + 1);
    init_dense_identity_matrix(H_tmp, m + 1, m);
    if (k == 0) copy_dense_matrix(H_tmp, H, m + 1, m);
    else dgemm_transpose2(Q, H, H_tmp, m + 1, m + 1, m);
    const double a = H_tmp[k * m + k], b = H_tmp[(k + 1) * m + k];
    const double J_denom = std::sqrt(std::fma(a, a, b * b));
    const double c_i = a / J_denom, s_i = b / J_denom;
    J[k * (m + 1) + k] = c_i;
    J[k * (m + 1) + k + 1] = s_i;
    J[(k + 1) * (m + 1) + k] = -1.0 * s_i;
    J[(k + 1) * (m + 1) + k + 1] = c_i;
    dgemm_transpose2(J, Q, Q_tmp, m + 1, m + 1, m + 1);
    copy_dense_matrix(Q, Q_tmp, m + 1, m + 1);
    dgemm_transpose2(Q, H, R, m + 1, m + 1, m);
}

// gmres.hpp:123-148
inline void update_g(int n_solver_iters, int restart_len, double *Q, double *g, double *g_tmp,
                     double &residual_norm, double beta) {
    const int m = restart_len;
    for (int i = 0; i <= m; ++i) g_tmp[i] = 0.0;
    g_tmp[0] = beta;
    for (int i = 0; i <= m; ++i) g[i] = g_tmp[i];
    dgemv(Q, g, g_tmp, m + 1, m + 1);
    for (int i = 0; i <= m; ++i) g[i] = g_tmp[i];
    residual_norm = std::abs(g[n_solver_iters + 1]);
}

// gmres.hpp:335-349: the k x k back-substitution R y = g of get_explicit_x
inline void back_substitution(int k, int m, const double *R, const double *g, double *y) {
    double diag_elem = 1.0;
    for (int row = k - 1; row >= 0; --row) {
        double sum = 0.0;
        for (int c = row; c < k; ++c) {
            if (row == c) diag_elem = R[row * m + c];
            else sum = std::fma(R[row * m + c], y[c], sum);
        }
        y[row] = (g[row] - sum) / diag_elem;
    }
}

class GMRESSolver : public Solver {
  public:
    double *x = nullptr, *x_old = nullptr, *V = nullptr, *Vy = nullptr, *w = nullptr;   // [dev]
    std::vector<double> y, H, H_tmp, J, Q, Q_tmp, R, g, g_tmp;                          // [host]
    double beta = 0.0;

    GMRESSolver(const Args *cli_args, Interface *device) : Solver(cli_args, device) {
        if (gmres_restart_len < 1 || gmres_restart_len > 64)
            bis_fatal("GMRES restart length must be in [1, 64]");
    }

    void allocate_structs(const int64_t n) override {
        Solver::allocate_structs(n);
        const int m = gmres_restart_len;
        x = dev_new(dev, n);
        x_old = dev_new(dev, n);
        V = dev_new(dev, n * (m + 1));
        Vy = dev_new(dev, n);
        w = dev_new(dev, n);
        y.assign(m + 1, 0.0);
        H.assign((m + 1) * m, 0.0);
        H_tmp.assign((m + 1) * m, 0.0);
        J.assign((m + 1) * (m + 1), 0.0);
        Q.assign((m + 1) * (m + 1), 0.0);
        Q_tmp.assign((m + 1) * (m + 1), 0.0);
        R.assign((m + 1) * m, 0.0);
        g.assign(m + 1, 0.0);
        g_tmp.assign(m + 1, 0.0);
    }

    // gmres.hpp:241-272
    void init_structs(const int64_t n) override {
        Solver::init_structs(n);
        const int m = gmres_restart_len;
        if (!gmres_restarted) {
            copy_vector(dev, x, x_0, n);
            copy_vector(dev, x_old, x_0, n);
        }
        init_vector(dev, V, 0.0, n * (m + 1));
        init_vector(dev, Vy, 0.0, n);
        init_vector(dev, w, 0.0, n);
        std::fill(y.begin(), y.end(), 0.0);
        std::fill(g.begin(), g.end(), 0.0);
        std::fill(g_tmp.begin(), g_tmp.end(), 0.0);
        std::fill(H.begin(), H.end(), 0.0);
        std::fill(H_tmp.begin(), H_tmp.end(), 0.0);
        std::fill(R.begin(), R.end(), 0.0);
        init_dense_identity_matrix(J.data(), m + 1, m + 1);
        init_dense_identity_matrix(Q.data(), m + 1, m + 1);
        init_dense_identity_matrix(Q_tmp.data(), m + 1, m + 1);
    }

    // gmres.hpp:274-324.  The stopping threshold comes from the UNpreconditioned
    // ||r0|| while the per-iteration residual is the preconditioned implicit one.
    void init_residual() override {
        BIS_OK(bis_spmv_residual(dev, dA->handle, x, b, residual, tmp, S_RR));
        if (!gmres_restarted) {
            residual_norm = std::sqrt(scalar(dev, S_RR));
            collected_residual_norms[collected_residual_norms_count++] = residual_norm;
        }
        precondition(residual, residual);
        BIS_OK(bis_sumsq_to_slot(dev, residual, N, S_BETA2));
        BIS_OK(bis_scale_inv_norm(dev, N, V, residual, S_BETA2));   // V[0] = residual * (1/beta)
        beta = std::sqrt(scalar(dev, S_BETA2));
        g[0] = beta;
        g_tmp[0] = beta;
        if (gmres_restarted) {
            residual_norm = beta;
            Solver::init_residual();
        }
    }

    // Device part of gmres_separate_iteration (gmres.hpp:150-183) for basis index k: everything it
    // needs (V[k]) is produced on the device, so it can be enqueued before the host has looked at
    // iteration k-1.  h_0k..h_kk land in slots S_H..S_H+k, ||w||^2 in S_H+k+1.
    void enqueue_iteration(const int k) {
        // V, w and the slots are fixed: the launches of basis index k are the same in every restart cycle
        graphed(k, [&] { enqueue_iteration_calls(k); });
    }
    void enqueue_iteration_calls(const int k) {
        spmv(dev, dA.get(), V + (int64_t)k * N, w);
        precondition(w, w);
        // orthogonalize_V: h_jk = (w, v_j) ; w -= h_jk v_j, j = 0..k ; h_{k+1,k} = ||w||
        BIS_OK(bis_dot_to_slot(dev, w, V, N, S_H));
        for (int j = 0; j <= k; ++j)
            BIS_OK(bis_mgs_step(dev, N, w, V + (int64_t)j * N, j < k ? V + (int64_t)(j + 1) * N : nullptr,
                                S_H + j, S_H + j + 1));
        BIS_OK(bis_scale_inv_norm(dev, N, V + (int64_t)(k + 1) * N, w, S_H + k + 1));
    }

    // gmres.hpp:150-196.  One split read fetches the Hessenberg column; inside a restart cycle the
    // device part of the NEXT iteration is enqueued behind that read, so the Givens update below runs
    // on the host while the device already works (it only writes w, V[k+2] and the scalar slots the
    // read has captured: harmless if this iteration turns out to be the last).
    bool ahead_ = false;
    void iterate(Timers *) override {
        const int m = gmres_restart_len;
        const int k = iter_count - gmres_restart_count * m;
        if (!ahead_) enqueue_iteration(k);
        ahead_ = false;
        BIS_OK(bis_scalar_read_begin(dev, S_H, k + 2));
        if (k + 1 < m && iter_count + 1 < max_iters - gmres_restart_count) {
            enqueue_iteration(k + 1);
            ahead_ = true;
        }
        double col[80];
        BIS_OK(bis_scalar_read_end(dev, S_H, k + 2, col));
        for (int j = 0; j <= k; ++j) H[k + j * m] = col[j];
        const double hn = std::sqrt(col[k + 1]);
        H[(k + 1) * m + k] = hn;   // a NaN norm is kept: the reference continues and stops on the NaN residual
        least_squares(k, m, J.data(), H.data(), H_tmp.data(), Q.data(), Q_tmp.data(), R.data());
        update_g(k, m, Q.data(), g.data(), g_tmp.data(), residual_norm, beta);
    }

    // gmres.hpp:326-375
    void get_explicit_x() override {
        const int m = gmres_restart_len;
        const int k = iter_count - gmres_restart_count * m;
        back_substitution(k, m, R.data(), g.data(), y.data());
        BIS_OK(bis_gmres_update_x(dev, N, k, V, y.data(), x, x_old, Vy));
    }

    void save_x_star() override {
        get_explicit_x();
        std::swap(x, x_star);
        Solver::save_x_star();
    }
    void record_residual_norm() override { Solver::record_residual_norm(); }

    // gmres.hpp:388-415
    void check_restart(Timers *timers) override {
        bool norm_convergence = residual_norm < stopping_criteria;
        bool over_max_iters = iter_count > max_iters;
        bool restart_cycle_reached = (iter_count % gmres_restart_len == 0) && (iter_count != 0);
        if (!norm_convergence && !over_max_iters && restart_cycle_reached) {
            gmres_restarted = true;
            ahead_ = false;
            get_explicit_x();
            copy_vector(dev, x_old, x, N);
            init_structs(N);
            init_residual();
            time_per_iteration[collected_residual_norms_count] = timers->per_iteration_time.check();
            ++gmres_restart_count;
        }
    }
    void exchange() override {}

    ~GMRESSolver() override {
        for (double **p : {&x, &x_old, &V, &Vy, &w}) dev_delete(dev, *p);
    }
};
