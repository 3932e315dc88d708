// On-device Krylov solve: MultiBlockSystem.solve (preconditioner/preconditioner.py:337-786)
// without PETSc.  GMRES(m) / FGMRES(m) / MINRES with PETSc's conventions as restated in
// oracle/krylov.py (SURVEY.md Appendix A.3): initial guess always non-zero (743), default
// convergence test against ||b|| (||P^-1 b|| for the preconditioned norm), classical
// Gram-Schmidt without refinement, iteration counter across restarts, max_it -> DIVERGED_ITS.
// Vectors never leave the device; per iteration the host reads the k+1 Gram-Schmidt
// scalars once (Hessenberg / Givens bookkeeping is host work on a handful of doubles).
#include <cmath>
#include <cstring>
#include <limits>

#include "krylov.cuh"

int ctl_solve_tf(ctl_handle_s *h, const double *b_tf, double *u_tf, const ctl_krylov_options *opts,
                    ctl_solve_result *result)
{
    if (!h->ks) h->ks = std::make_shared<KrylovState>();
    CTL_CHECK(opts->ksp_type >= CTL_KSP_GMRES && opts->ksp_type <= CTL_KSP_MINRES, CTL_ERR_ARG,
              "ctl_solve: unknown ksp_type");
    CTL_CHECK(opts->pc >= CTL_PC_NONE && opts->pc <= CTL_PC_CALLBACK, CTL_ERR_ARG, "ctl_solve: unknown pc kind");
    if (opts->pc == CTL_PC_BUILTIN)
        CTL_CHECK(h->pc && h->pc->ready, CTL_ERR_STATE, "ctl_solve: call ctl_pc_setup first");
    Solver K(h, *opts, *result, *h->ks, h->pool, h->vec_len(), "ctl_solve", h->pc_cb, h->pc_cb_user);
    return krylov_solve(K, b_tf, u_tf);
}

extern "C" {

int ctl_krylov_default_options(ctl_krylov_options *o)
{
    if (!o) return CTL_ERR_ARG;
    o->ksp_type = CTL_KSP_FGMRES;      // solver_parameters.get("linear_solver", "fgmres"), preconditioner.py:733
    o->restart = 30;                   // PETSc default; only "gmres_restart" overrides it (747-748)
    o->max_it = 1000;                  // 742
    o->pc = CTL_PC_NONE;
    o->rtol = 1e-5;
    o->atol = 1e-50;
    o->divtol = 1e4;
    return CTL_OK;
}

int ctl_solve(ctl_handle h, const double *b, double *u, int layout, const ctl_krylov_options *opts,
              ctl_solve_result *result)
{
    CTL_CHECK(h && b && u && opts && result, CTL_ERR_ARG, "ctl_solve: null argument");
    CTL_CHECK(h->assembled, CTL_ERR_STATE, "ctl_solve: ctl_assemble has not been called");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    if (layout == CTL_LAYOUT_TIME_FASTEST) return ctl_solve_tf(h, b, u, opts, result);
    return with_tf(h, layout, {b, u}, u,
                   [&](const double *bt, double *ut) { return ctl_solve_tf(h, bt, ut, opts, result); });
}

int ctl_solve_host(ctl_handle h, const double *b_host, double *u_host, const ctl_krylov_options *opts,
                   ctl_solve_result *result)
{
    CTL_CHECK(h && b_host && u_host && opts && result, CTL_ERR_ARG, "ctl_solve_host: null argument");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    const size_t bytes = (size_t)ctl_vec_len(h, CTL_LAYOUT_BLOCK_MAJOR) * sizeof(double);
    Scratch b, u;     // scratch vectors are at least block-major sized
    CTL_TRY(h->pool.take(&b));
    CTL_TRY(h->pool.take(&u));
    if (cudaMemcpyAsync(b, b_host, bytes, cudaMemcpyHostToDevice, h->stream) != cudaSuccess ||
        cudaMemcpyAsync(u, u_host, bytes, cudaMemcpyHostToDevice, h->stream) != cudaSuccess) {
        ctl_set_error(h, "ctl_solve_host: host to device copy failed");
        return CTL_ERR_CUDA;
    }
    CTL_TRY(ctl_solve(h, b, u, CTL_LAYOUT_BLOCK_MAJOR, opts, result));
    if (cudaMemcpyAsync(u_host, u, bytes, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess ||
        cudaStreamSynchronize(h->stream) != cudaSuccess) {
        ctl_set_error(h, "ctl_solve_host: device to host copy failed");
        return CTL_ERR_CUDA;
    }
    return CTL_OK;
}

int ctl_kkt_residual_norm(ctl_handle h, const double *b, const double *x, int layout, double *out)
{
    CTL_CHECK(h && b && x && out, CTL_ERR_ARG, "ctl_kkt_residual_norm: null argument");
    CTL_CHECK(h->assembled, CTL_ERR_STATE, "ctl_kkt_residual_norm: ctl_assemble has not been called");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    const int64_t len = h->vec_len();
    return with_tf(h, layout, {b, x, nullptr}, nullptr, [&](double *bt, const double *xt, double *r) {
        if (h->d_bc_rows_all) {
            const size_t panel = (size_t)h->n_loc * h->ld;
            CTL_TRY(pcb_bc_fixup(h, h->d_bc_rows_all, h->n_bc_all, nullptr, bt));
            CTL_TRY(pcb_bc_fixup(h, h->d_bc_rows_all, h->n_bc_all, nullptr, bt + panel));
        }
        CTL_TRY(ctl_kkt_apply_tf(h, xt, r));
        CTL_TRY(vec_lincomb(h, r, 1.0, bt, -1.0, r, 0.0, nullptr, nullptr, len));
        return vec_norm_host(h, r, len, out);
    });
}

// Residual of the outer Picard / Gauss-Newton loop on device vectors.  non_linear_res_eval (control/control.py:
// 2442-2818) assembles it row by row from 2 n_t FE mat-vecs; after the T_1 / T_2 transforms that linear_solve
// applies to ready right-hand sides it EQUALS b - A x with b the right-hand side of linear_solve for the data and
// A the operator with D_v at the iterate (tests/test_oracle.py::test_non_linear_residual_is_rhs_minus_operator), so
// it is one fused operator apply and one vector update here, and doubles as the right-hand side of the increment
// solve.  The norm the loop tests is that of the UNtransformed residual: ||T^-1 r||.
int ctl_nonlinear_residual(ctl_handle h, const double *b, const double *x, double *r_out, int layout, double *norm_host)
{
    CTL_CHECK(h && b && x && r_out && norm_host, CTL_ERR_ARG, "ctl_nonlinear_residual: null argument");
    CTL_CHECK(h->assembled, CTL_ERR_STATE, "ctl_nonlinear_residual: ctl_assemble has not been called");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    const int64_t len = h->vec_len();
    const size_t panel = (size_t)h->n_loc * h->ld;
    return with_tf(h, layout, {b, x, nullptr}, nullptr, [&](const double *bt, const double *xt, double *r) {
        CTL_TRY(ctl_kkt_apply_tf(h, xt, r));
        CTL_TRY(vec_lincomb(h, r, 1.0, bt, -1.0, r, 0.0, nullptr, nullptr, len));
        if (h->d_bc_rows_all) {      // rows of constrained dofs carry no residual (2816-2817)
            CTL_TRY(pcb_bc_fixup(h, h->d_bc_rows_all, h->n_bc_all, nullptr, r));
            CTL_TRY(pcb_bc_fixup(h, h->d_bc_rows_all, h->n_bc_all, nullptr, r + panel));
        }
        CTL_TRY((layout == CTL_LAYOUT_TIME_FASTEST) ? vec_copy(h, r_out, r, len) : ctl_to_bm(h, r, r_out));
        if (h->cfg.CN) {
            CTL_TRY(ctl_panel_tinv(h, r, 1, h->n_loc));
            CTL_TRY(ctl_panel_tinv(h, r + panel, 2, h->n_loc));
        }
        return vec_norm_host(h, r, len, norm_host);
    });
}

// J_h (SURVEY.md section 8c), evaluated on the host from the mass matrix the caller handed over
int ctl_objective_host(ctl_handle h, const double *v, const double *zeta, const double *v_hat, double *out)
{
    CTL_CHECK(h && v && zeta && v_hat && out, CTL_ERR_ARG, "ctl_objective_host: null argument");
    CTL_CHECK(!h->h_M.empty(), CTL_ERR_STATE, "ctl_objective_host: no mass matrix");
    const int n = h->n, n_t = h->cfg.n_t;
    const double tau = h->cfg.tau, beta = h->cfg.beta;
    std::vector<double> d(n);
    auto quad = [&](const double *x) {
        double s = 0.0;
        for (int r = 0; r < n; ++r) {
            double a = 0.0;
            for (int k = h->h_indptr[r]; k < h->h_indptr[r + 1]; ++k) a += h->h_M[k] * x[h->h_indices[k]];
            s += x[r] * a;
        }
        return s;
    };
    double J = 0.0;
    for (int i = 0; i < n_t; ++i) {
        const double w = (h->cfg.CN && (i == 0 || i == n_t - 1)) ? 0.5 * tau : tau;
        for (int r = 0; r < n; ++r) d[r] = v[(size_t)i * n + r] - v_hat[(size_t)i * n + r];
        J += 0.5 * w * quad(d.data());
        J += 0.5 / beta * w * quad(zeta + (size_t)i * n);
    }
    *out = J;
    return CTL_OK;
}

}  // extern "C"
