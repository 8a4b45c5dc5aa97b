// host/host_capi.cpp -- C entry points of the HOST library (libbis_host.so):
// the reference-shaped Solver/harness stack driven from plain C (ctypes in the
// tests and bench.py).  Device work goes through the C-ABI of libbis_b200.so.
#include "lu_factors.hpp"
#include "run.hpp"

#include <cstring>

static thread_local std::string g_host_err;

extern "C" {

const char *bis_host_last_error(void) { return g_host_err.c_str(); }

// parse_cli round trip (CPU-only test of the host logic): fills
// out[0]=method, out[1]=precond, out[2]=restart_length, out[3]=num_scale.
int bis_host_parse_cli(int argc, char **argv, int *out) {
    try {
        Args a;
        parse_cli(&a, argc, argv);
        out[0] = static_cast<int>(a.method);
        out[1] = static_cast<int>(a.preconditioner);
        out[2] = a.restart_length;
        out[3] = a.num_scale ? 1 : 0;
        return 0;
    } catch (const std::exception &e) {
        g_host_err = e.what();
        return 1;
    }
}

// Host preprocessing (CPU-only testable): strict split + diagonals (+ ILU(0)).
// Call with l_col == NULL to obtain the sizes first.
int bis_host_factor(int n, const int *rp, const int *col, const double *val, int precond, int *l_rp,
                    int *l_col, double *l_val, int *u_rp, int *u_col, double *u_val, double *A_D,
                    double *A_D_inv, double *L_D, double *U_D) {
    try {
        MatrixCRS A(n, n, rp[n]);
        std::memcpy(A.row_ptr, rp, sizeof(int) * (n + 1));
        std::memcpy(A.col, col, sizeof(int) * rp[n]);
        std::memcpy(A.val, val, sizeof(double) * rp[n]);
        MatrixCRS L, U;
        std::vector<double> d(n, 1.0), di(n, 0.0), ld(n, 1.0), ud(n, 1.0);
        factor_LU(&A, d.data(), di.data(), &L, ld.data(), &U, ud.data(), static_cast<PrecondType>(precond));
        std::memcpy(l_rp, L.row_ptr, sizeof(int) * (n + 1));
        std::memcpy(u_rp, U.row_ptr, sizeof(int) * (n + 1));
        if (l_col) {
            std::memcpy(l_col, L.col, sizeof(int) * L.nnz);
            std::memcpy(l_val, L.val, sizeof(double) * L.nnz);
            std::memcpy(u_col, U.col, sizeof(int) * U.nnz);
            std::memcpy(u_val, U.val, sizeof(double) * U.nnz);
            std::memcpy(A_D, d.data(), sizeof(double) * n);
            std::memcpy(A_D_inv, di.data(), sizeof(double) * n);
            std::memcpy(L_D, ld.data(), sizeof(double) * n);
            std::memcpy(U_D, ud.data(), sizeof(double) * n);
        }
        return 0;
    } catch (const std::exception &e) {
        g_host_err = e.what();
        return 1;
    }
}

// Host matrix generators / reader (CPU-only testable).  kind 0: .mtx path in
// `name`; otherwise a generator name.  Two-phase: sizes, then fill.
static std::unique_ptr<MatrixCRS> g_mat;
int bis_host_matrix_begin(const char *name, int *n, int *nnz) {
    try {
        Args a;
        a.matrix_file_name = name;
        std::unique_ptr<DeviceCRS> none;
        obtain_matrix(&a, nullptr, g_mat, none, /*on_host=*/true);
        *n = g_mat->n_rows;
        *nnz = g_mat->nnz;
        return 0;
    } catch (const std::exception &e) {
        g_host_err = e.what();
        return 1;
    }
}
int bis_host_matrix_fetch(int *rp, int *col, double *val) {
    if (!g_mat) return 1;
    std::memcpy(rp, g_mat->row_ptr, sizeof(int) * (g_mat->n_rows + 1));
    std::memcpy(col, g_mat->col, sizeof(int) * g_mat->nnz);
    std::memcpy(val, g_mat->val, sizeof(double) * g_mat->nnz);
    g_mat.reset();
    return 0;
}

// The harness loop driven by a device-free solver that only records the order of the calls (CPU-only
// test of solve() / harness_step: run-ahead order, no speculation past max_iters, stop decisions).
// The k-th residual norm is r0 * decay^k.  trace: 'I' iterate, 'b' norm readback enqueued, 'e' norm
// waited for, 's' synchronous sample, 'X' exchange, 'R' check_restart, '|' end of a loop pass.
namespace {
class TraceSolver : public Solver {
  public:
    std::string trace;
    bool ahead_ok;
    double r0, decay;
    int iterates = 0;
    TraceSolver(const Args *a, bool run_ahead, double r0_, double decay_)
        : Solver(a, nullptr), ahead_ok(run_ahead), r0(r0_), decay(decay_) {}
    void iterate(Timers *) override { trace += 'I'; ++iterates; }
    void exchange() override { trace += 'X'; }
    void check_restart(Timers *) override { trace += "R|"; }
    bool can_run_ahead() const override { return ahead_ok; }
    void read_norm_begin() override { trace += 'b'; }
    double read_norm_end() override {
        trace += 'e';
        const double r = r0 * std::pow(decay, iter_count);
        return r * r;
    }
    void record_residual_norm() override {
        trace += 's';
        residual_norm = r0 * std::pow(decay, iter_count);
        Solver::record_residual_norm();
    }
    void save_x_star() override {}
};
} // namespace

int bis_host_harness_trace(int run_ahead, int max_iters, double tol, double decay, char *trace, int trace_cap,
                           int *out) {
    try {
        Args args;
        args.quiet = true;
        TraceSolver s(&args, run_ahead != 0, 1.0, decay);
        if (max_iters > MAX_ITERS) bis_fatal("max_iters exceeds MAX_ITERS");
        s.max_iters = max_iters;
        s.tolerance = tol;
        s.residual_norm = 1.0;
        s.collected_residual_norms[s.collected_residual_norms_count++] = 1.0;   // init_residual
        s.init_stopping_criteria();
        Timers timers;
        solve(&args, &s, &timers);
        std::snprintf(trace, (size_t)trace_cap, "%s", s.trace.c_str());
        out[0] = s.iter_count;
        out[1] = s.iterates;
        out[2] = s.convergence_flag ? 1 : 0;
        out[3] = s.collected_residual_norms_count;
        return 0;
    } catch (const std::exception &e) {
        g_host_err = e.what();
        return 1;
    }
}

// GMRES host pieces (CPU-only testable against the oracle).
void bis_host_gmres_least_squares(int k, int m, double *J, double *H, double *H_tmp, double *Q,
                                  double *Q_tmp, double *R) {
    least_squares(k, m, J, H, H_tmp, Q, Q_tmp, R);
}
double bis_host_gmres_update_g(int k, int m, double *Q, double *g, double *g_tmp, double beta) {
    double rn = 0.0;
    update_g(k, m, Q, g, g_tmp, rn, beta);
    return rn;
}

// A whole solve on the device.  Matrix: host CRS arrays (rp != NULL) or a
// generator / file name.  b / x0: host vectors or NULL (B_VAL / INIT_X_VAL).
// max_iters <= 0 keeps MAX_ITERS; tol <= 0 keeps TOL.
// history: 2*MAX_ITERS doubles; iter_time likewise (may be NULL); x_star: n
// doubles (may be NULL).
// out_int: iter_count, history count, converged, restart_count, kernel launches.
// out_dbl: stopping criteria, final true residual, solve seconds, preprocessing
// seconds, mean seconds per iteration (harness table, first iteration excluded).
int bis_host_solve(bis_context *dev, const char *matrix_name, int n, const int *rp, const int *col,
                   const double *val, int method, int precond, int restart_len, const double *b,
                   const double *x0, int max_iters, double tol, int quiet, int num_scale, double *history,
                   double *iter_time, double *x_star, int *out_int, double *out_dbl) {
    try {
        Args args;
        args.matrix_file_name = matrix_name ? matrix_name : "in-memory";
        args.method = static_cast<SolverType>(method);
        args.preconditioner = static_cast<PrecondType>(precond);
        args.restart_length = restart_len;
        args.quiet = quiet != 0;
        args.num_scale = num_scale != 0;
        Timers timers;
        std::unique_ptr<Solver> solver = make_solver(&args, dev);
        if (max_iters > 0) {
            if (max_iters > MAX_ITERS) bis_fatal("max_iters exceeds MAX_ITERS");
            solver->max_iters = max_iters;
        }
        if (tol > 0) solver->tolerance = tol;
        std::unique_ptr<MatrixCRS> A;
        std::unique_ptr<DeviceCRS> dA;
        if (rp) {
            A = std::make_unique<MatrixCRS>(n, n, rp[n]);
            std::memcpy(A->row_ptr, rp, sizeof(int) * (n + 1));
            std::memcpy(A->col, col, sizeof(int) * rp[n]);
            std::memcpy(A->val, val, sizeof(double) * rp[n]);
        } else {
            obtain_matrix(&args, dev, A, dA);
        }
        int64_t info0[8];
        BIS_OK(bis_context_info(dev, info0));
        TIME(timers.preprocessing, preprocessing(&args, solver.get(), &timers, A, std::move(dA), b, x0))
        TIME(timers.solve, solve(&args, solver.get(), &timers))
        int64_t info1[8];
        BIS_OK(bis_context_info(dev, info1));
        const int cnt = solver->collected_residual_norms_count;
        const int ncopy = std::min(cnt + 2, 2 * MAX_ITERS);
        for (int i = 0; i < ncopy; ++i) {
            history[i] = solver->collected_residual_norms[i];
            if (iter_time) iter_time[i] = solver->time_per_iteration[i];
        }
        if (x_star) BIS_OK(bis_vector_download(dev, x_star, solver->x_star, solver->N));
        out_int[0] = solver->iter_count;
        out_int[1] = cnt;
        out_int[2] = solver->convergence_flag ? 1 : 0;
        out_int[3] = solver->gmres_restart_count;
        out_int[4] = (int)(info1[3] - info0[3]);
        out_dbl[0] = solver->stopping_criteria;
        out_dbl[1] = solver->residual_norm;
        out_dbl[2] = timers.solve_time.get_wtime();
        out_dbl[3] = timers.preprocessing_time.get_wtime();
        double acc = 0.0;
        int m = 0;
        for (int i = 3; i <= cnt; ++i) {   // time_per_iteration[i+1] pairs with history[i]; skip the first
            acc += solver->time_per_iteration[i];
            ++m;
        }
        out_dbl[4] = m ? acc / m : 0.0;
        if (!quiet) postprocessing(&args, solver.get(), &timers);
        return 0;
    } catch (const std::exception &e) {
        g_host_err = e.what();
        return 1;
    }
}


// ---- measurement sessions (bench.py) ----------------------------------------------
// A session owns one Solver on one named matrix.  Two timed regions:
//  * e2e: what a user of the host stack does -- host b / x0 arrays in,
//    preprocessing() (allocate, upload, init_residual), solve() for exactly
//    `steps` iterations (the harness reads the residual norm back every
//    iteration), x_star downloaded to host memory.  Wall clock, device idle on
//    both sides.  Matrix generation is outside (the matrix is the operator).
//  * resident: state already in HBM; `warmup` untimed iterations of the
//    harness loop body, then `steps` timed ones between two CUDA events on the
//    context's stream.
struct BenchSession {
    Args args;
    Timers timers;
    std::unique_ptr<Solver> solver;
    bis_context *dev = nullptr;
    double setup_ms = 0.0;   // wall time of the last obtain_matrix (generation + SpMV tile format + order table)
};

static void bench_make(BenchSession *s) {
    s->solver = make_solver(&s->args, s->dev);
}

void *bis_host_bench_open(bis_context *dev, const char *matrix_name, int method, int precond,
                          int restart_len) {
    try {
        auto s = std::make_unique<BenchSession>();
        s->dev = dev;
        s->args.matrix_file_name = matrix_name;
        s->args.method = static_cast<SolverType>(method);
        s->args.preconditioner = static_cast<PrecondType>(precond);
        s->args.restart_length = restart_len;
        s->args.quiet = true;
        return s.release();
    } catch (const std::exception &e) {
        g_host_err = e.what();
        return nullptr;
    }
}

void bis_host_bench_close(void *h) { delete static_cast<BenchSession *>(h); }

// info: [0] local rows, [1] global rows, [2] local nnz, [3] global nnz, [4] row_ptr bytes
static void bench_fill_info(Solver *solver, int64_t *info) {
    int64_t mi[8];
    BIS_OK(bis_matrix_info(solver->dA->handle, mi));
    info[0] = mi[0]; info[1] = mi[1]; info[2] = mi[2]; info[3] = mi[3]; info[4] = mi[4];
}

// out: [0] wall ms of the whole region, [1] iterations done, [2] kernel launches,
//      [3] last residual norm, [4] ||r0||, [5] final true residual
int bis_host_bench_e2e(void *h, int steps, const double *b_host, const double *x0_host,
                       double *x_star_host, double *out, int64_t *info) {
    auto *s = static_cast<BenchSession *>(h);
    try {
        if (steps > MAX_ITERS) bis_fatal("bench: steps outside [1, MAX_ITERS]");
        bench_make(s);
        Solver *solver = s->solver.get();
        if (steps >= 1) {
            solver->max_iters = steps;
            solver->tolerance = 0.0;   // never stop early: exactly `steps` iterations
        }                              // steps <= 0: a real solve (TOL, MAX_ITERS)
        std::unique_ptr<MatrixCRS> A;
        std::unique_ptr<DeviceCRS> dA;
        Stopwatch ws;
        ws.start();
        obtain_matrix(&s->args, s->dev, A, dA);
        BIS_OK(bis_context_synchronize(s->dev));
        s->setup_ms = ws.check() * 1e3;
        int64_t i0[8], i1[8];
        BIS_OK(bis_context_info(s->dev, i0));
        Stopwatch w;
        w.start();
        s->timers = Timers();
        preprocessing(&s->args, solver, &s->timers, A, std::move(dA), b_host, x0_host);
        const double t_pre = w.check();
        solve(&s->args, solver, &s->timers);
        const double t_solve = w.check();
        if (x_star_host) BIS_OK(bis_vector_download(s->dev, x_star_host, solver->x_star, solver->N));
        BIS_OK(bis_context_synchronize(s->dev));
        out[0] = w.check() * 1e3;
        // breakdown of the wall time (ms): allocate + init + uploads | r0 and factor step | loop | x_star download
        out[6] = s->timers.preprocessing_init_time.get_wtime() * 1e3;
        out[7] = (t_pre - s->timers.preprocessing_init_time.get_wtime()) * 1e3;
        info[6] = (int64_t)((t_solve - t_pre) * 1e6);
        info[7] = (int64_t)((w.check() - t_solve) * 1e6);
        BIS_OK(bis_context_info(s->dev, i1));
        out[1] = solver->iter_count;
        out[2] = (double)(i1[3] - i0[3]);
        out[3] = solver->collected_residual_norms[solver->collected_residual_norms_count - 1];
        out[4] = solver->collected_residual_norms[0];
        out[5] = solver->residual_norm;
        bench_fill_info(solver, info);
        return 0;   // the solver stays alive until the next call (bis_host_bench_history)
    } catch (const std::exception &e) {
        g_host_err = e.what();
        s->solver.reset();
        return 1;
    }
}

double bis_host_bench_setup_ms(void *h) { return static_cast<BenchSession *>(h)->setup_ms; }

// History of the session's solver: the first `cap` collected residual norms; returns how many exist.
int bis_host_bench_history(void *h, double *out, int cap) {
    auto *s = static_cast<BenchSession *>(h);
    if (!s->solver) return 0;
    const int n = s->solver->collected_residual_norms_count;
    for (int i = 0; i < n && i < cap; ++i) out[i] = s->solver->collected_residual_norms[i];
    return n;
}

// Untimed: build the solver, obtain the matrix, preprocessing, `warmup` iterations.
int bis_host_bench_prepare(void *h, int warmup, int64_t *info) {
    auto *s = static_cast<BenchSession *>(h);
    try {
        bench_make(s);
        Solver *solver = s->solver.get();
        solver->tolerance = 0.0;
        std::unique_ptr<MatrixCRS> A;
        std::unique_ptr<DeviceCRS> dA;
        obtain_matrix(&s->args, s->dev, A, dA);
        preprocessing(&s->args, solver, &s->timers, A, std::move(dA));
        bool ahead = false;
        for (int i = 0; i < warmup; ++i) harness_step(solver, &s->timers, ahead, i + 1 < warmup);
        BIS_OK(bis_context_synchronize(s->dev));
        bench_fill_info(solver, info);
        return 0;
    } catch (const std::exception &e) {
        g_host_err = e.what();
        s->solver.reset();
        return 1;
    }
}

// Timed: exactly `steps` iterations of the harness loop body (solver_harness.hpp:17-50).
// out: [0] device ms (CUDA events on the context's stream), [1] wall ms, [2] kernel
// launches, [3] residual norm after the last iteration, [4] ||r0||
int bis_host_bench_run(void *h, int steps, double *out) {
    auto *s = static_cast<BenchSession *>(h);
    try {
        Solver *solver = s->solver.get();
        if (!solver) bis_fatal("bench: prepare first");
        if (solver->iter_count + steps + 1 >= MAX_ITERS) bis_fatal("bench: warmup + steps exceed MAX_ITERS");
        int64_t i0[8], i1[8];
        BIS_OK(bis_context_info(s->dev, i0));
        BIS_OK(bis_dist_stream_barrier(s->dev));   // all ranks' streams start the timed region together
        Stopwatch w;
        w.start();
        BIS_OK(bis_timer_start(s->dev));
        // the loop body of solve(); the last timed step does not run ahead, so exactly `steps` iterations
        // are enqueued between the two timer events
        bool ahead = false;
        for (int i = 0; i < steps; ++i) harness_step(solver, &s->timers, ahead, i + 1 < steps);
        double ms = 0.0;
        BIS_OK(bis_timer_stop(s->dev, &ms));
        out[1] = w.check() * 1e3;
        out[0] = ms;
        BIS_OK(bis_context_info(s->dev, i1));
        out[2] = (double)(i1[3] - i0[3]);
        out[3] = solver->residual_norm;
        out[4] = solver->collected_residual_norms[0];
        return 0;
    } catch (const std::exception &e) {
        g_host_err = e.what();
        return 1;
    }
}

// Enqueues a copy of the current iterate of a CG session (x after the last step run: what save_x_star() would
// hand back) into the device vector x_dev of the session's local rows.  The session's state is not touched.
int bis_host_bench_copy_x(void *h, double *x_dev) {
    auto *s = static_cast<BenchSession *>(h);
    try {
        auto *cg = dynamic_cast<ConjugateGradientSolver *>(s->solver.get());
        if (!cg) bis_fatal("bench: copy_x needs a prepared CG session");
        copy_vector(s->dev, x_dev, cg->x_old, cg->N);
        return 0;
    } catch (const std::exception &e) {
        g_host_err = e.what();
        return 1;
    }
}

} // extern "C"
