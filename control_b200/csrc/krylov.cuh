// Krylov methods shared by the heat-type KKT solve (krylov.cu) and the Stokes outer solve
// (stokes.cu): see krylov.cu for the conventions restated from PETSc.
#pragma once
#include <cmath>
#include <cstring>
#include <limits>

#include "common.cuh"
#include "pc.cuh"
#include "vec_ops.cuh"

struct KrylovState {
    std::vector<double *> basis;      // V_0..V_m then Z_0..Z_{m-1}
    std::vector<EventPair> events;    // one pair per timed operator / pc application of a solve
    size_t next_event = 0;
    std::vector<std::pair<size_t, int>> spans;   // (event pair, 0 = mult / 1 = pc)
    KrylovState() = default;
    KrylovState(const KrylovState &) = delete;
    KrylovState &operator=(const KrylovState &) = delete;
    ~KrylovState()
    {
        for (double *p : basis) cudaFree(p);
    }
};

namespace {

struct Conv {   // KSPConvergedDefault
    double rtol, atol, divtol, ttol, rnorm0;
    Conv(double rtol_, double atol_, double divtol_, double ref)
        : rtol(rtol_), atol(atol_), divtol(divtol_), ttol(std::max(rtol_ * ref, atol_)), rnorm0(ref) {}
    int operator()(double rnorm) const
    {
        if (!std::isfinite(rnorm)) return CTL_DIVERGED_NANORINF;
        if (rnorm <= ttol) return rnorm < atol ? CTL_CONVERGED_ATOL : CTL_CONVERGED_RTOL;
        if (rnorm >= divtol * rnorm0) return CTL_DIVERGED_DTOL;
        return 0;
    }
};

struct Solver {
    ctl_handle_s *h;
    const ctl_krylov_options &o;
    ctl_solve_result &res;
    KrylovState &ks;
    ScratchPool &pool;          // vectors of length len
    int64_t len;
    const char *name;           // entry point, for the error messages
    ctl_pc_callback cb;         // pc = CTL_PC_CALLBACK: the user's pc_fn on block-major vectors
    void *cb_user;

    // h carries the stream, the reduction workspace and the error string; the linear system
    // itself is behind the virtual hooks (defaults: the heat-type KKT system of the handle)
    Solver(ctl_handle_s *h_, const ctl_krylov_options &o_, ctl_solve_result &r_, KrylovState &ks_, ScratchPool &pool_,
           int64_t len_, const char *name_, ctl_pc_callback cb_, void *cb_user_)
        : h(h_), o(o_), res(r_), ks(ks_), pool(pool_), len(len_), name(name_), cb(cb_), cb_user(cb_user_) {}

    virtual ~Solver() {}

    virtual int apply_operator(const double *x, double *y) { return ctl_kkt_apply_tf(h, x, y); }
    virtual int apply_builtin_pc(const double *x, double *y) { return ctl_pc_apply_tf(h, x, y); }
    virtual int to_bm(const double *tf, double *bm) { return ctl_to_bm(h, tf, bm); }
    virtual int to_tf(const double *bm, double *tf) { return ctl_to_tf(h, bm, tf); }

    int span_begin(int kind)
    {
        if (ks.next_event == ks.events.size()) {
            EventPair e;
            CTL_TRY(e.create(h));
            ks.events.push_back(std::move(e));
        }
        ks.spans.emplace_back(ks.next_event, kind);
        CTL_CUDA(cudaEventRecord(ks.events[ks.next_event].begin, h->stream));
        return CTL_OK;
    }

    int span_end()
    {
        CTL_CUDA(cudaEventRecord(ks.events[ks.next_event].end, h->stream));
        ks.next_event++;
        return CTL_OK;
    }

    int op(const double *x, double *y)
    {
        res.n_mult++;
        CTL_TRY(span_begin(0));
        CTL_TRY(apply_operator(x, y));
        return span_end();
    }

    // Preconditioner.apply (preconditioner/preconditioner.py:562-656)
    int prec(const double *x, double *y)
    {
        res.n_pc++;
        CTL_TRY(span_begin(1));
        if (o.pc == CTL_PC_NONE) {
            CTL_TRY(vec_copy(h, y, x, len));       // pc_fn = None: u = b (342-345)
        } else if (o.pc == CTL_PC_BUILTIN) {
            CTL_TRY(apply_builtin_pc(x, y));
        } else {
            CTL_TRY(apply_callback_pc(x, y));
        }
        return span_end();
    }

    // Preconditioner.apply around a user pc_fn (preconditioner/preconditioner.py:562-656): project the right-hand
    // side, hand block-major device vectors of the system to the callback, restore the constrained entries
    int apply_callback_pc(const double *x, double *y)
    {
        CTL_CHECK(cb, CTL_ERR_STATE, std::string(name) + ": no preconditioner callback installed");
        Scratch bm_b, bm_u, xc;
        for (Scratch *s : {&bm_b, &bm_u, &xc}) CTL_TRY(pool.take(s));
        CTL_TRY(vec_copy(h, xc, x, len));
        CTL_TRY(project(xc, nullptr));                  // pc_pre_mult_corrected
        CTL_TRY(to_bm(xc, bm_b));
        CTL_TRY(vec_zero(h, bm_u, len));
        cudaStreamSynchronize(h->stream);
        if (cb(cb_user, bm_b, bm_u) != 0) {
            ctl_set_error(h, "preconditioner callback failed");
            return CTL_ERR_CALLBACK;
        }
        CTL_TRY(to_tf(bm_u, y));
        return project(y, x);                           // pc_post_mult_correct
    }

    // constrained rows of both panels: v = wrap ? wrap : 0
    virtual int project(double *v, const double *wrap)
    {
        if (!h->d_bc_rows_all) return CTL_OK;
        const size_t panel = (size_t)h->n_loc * h->ld;
        CTL_TRY(pcb_bc_fixup(h, h->d_bc_rows_all, h->n_bc_all, wrap, v));
        return pcb_bc_fixup(h, h->d_bc_rows_all, h->n_bc_all, wrap ? wrap + panel : nullptr, v + panel);
    }

    int norm(const double *x, double *out) { return vec_norm_host(h, x, len, out); }
    int dot(const double *x, const double *y, double *out) { return vec_dot_host(h, x, y, len, out); }

    void record(double rnorm)
    {
        res.rnorm = rnorm;
        if (res.n_history < CTL_HISTORY_MAX) res.history[res.n_history++] = rnorm;
    }

    int ensure_basis(size_t count)
    {
        while (ks.basis.size() < count) {
            double *p = nullptr;
            CTL_CUDA(cudaMalloc((void **)&p, (size_t)len * sizeof(double)));
            ks.basis.push_back(p);
        }
        return CTL_OK;
    }

    int gmres(const double *b, double *x)
    {
        const bool flexible = o.ksp_type == CTL_KSP_FGMRES;
        // a restart length beyond max_it is never reached: do not allocate basis vectors for it
        const int m = std::max(1, std::min(o.restart, std::max(1, o.max_it)));
        CTL_CHECK(m + 3 <= 256, CTL_ERR_ARG, "ctl_solve: gmres_restart above 253 is not supported");
        CTL_TRY(ensure_basis((size_t)(m + 1) + (flexible ? m : 0)));
        double **V = ks.basis.data();
        double **Z = ks.basis.data() + (m + 1);
        Scratch t;
        CTL_TRY(pool.take(&t));
        double *partials, *scal;
        CTL_TRY(vec_workspace(h, &partials, &scal));
        double ref = 0.0;
        if (flexible) {
            CTL_TRY(norm(b, &ref));
        } else {
            CTL_TRY(prec(b, t));
            CTL_TRY(norm(t, &ref));
        }
        res.ref_norm = ref;
        const Conv conv(o.rtol, o.atol, o.divtol, ref);
        std::vector<double> H((size_t)(m + 1) * m), g(m + 1), cs(m), sn(m), hcol(m + 2);
        while (res.reason == 0) {
            // r = b - A x (left PC: P^-1 (b - A x)) -> V[0]
            CTL_TRY(op(x, t));
            if (flexible) {
                CTL_TRY(vec_lincomb(h, V[0], 1.0, b, -1.0, t, 0.0, nullptr, nullptr, len));
            } else {
                CTL_TRY(vec_lincomb(h, t, 1.0, b, -1.0, t, 0.0, nullptr, nullptr, len));
                CTL_TRY(prec(t, V[0]));
            }
            double rnorm = 0.0;
            CTL_TRY(norm(V[0], &rnorm));
            if (res.its == 0) record(rnorm);
            res.reason = conv(rnorm);
            if (res.reason) break;
            if (rnorm == 0.0) {
                res.reason = CTL_CONVERGED_ATOL;
                break;
            }
            CTL_TRY(vec_lincomb(h, V[0], 1.0 / rnorm, V[0], 0.0, nullptr, 0.0, nullptr, nullptr, len));
            std::fill(H.begin(), H.end(), 0.0);
            std::fill(g.begin(), g.end(), 0.0);
            g[0] = rnorm;
            int it = 0;
            while (res.reason == 0 && it < m && res.its < o.max_it) {
                double *w = V[it + 1];
                if (flexible) {
                    CTL_TRY(prec(V[it], Z[it]));
                    CTL_TRY(op(Z[it], w));
                } else {
                    CTL_TRY(op(V[it], t));
                    CTL_TRY(prec(t, w));
                }
                // classical Gram-Schmidt: all dots against the unmodified w, one update, norm
                CTL_TRY(vec_multi_dot_dev(h, V, it + 1, w, len, scal, nullptr));
                CTL_TRY(vec_maxpy_dev(h, w, V, it + 1, scal, -1.0, len, scal + it + 1, scal + it + 2));
                CTL_TRY(vec_read_scalars(h, scal, it + 3, hcol.data()));
                const double tt = hcol[it + 2];
                for (int k = 0; k <= it; ++k) H[(size_t)k * m + it] = hcol[k];
                H[(size_t)(it + 1) * m + it] = tt;
                const bool happy = tt == 0.0;
                if (!happy) CTL_TRY(vec_lincomb(h, w, 1.0 / tt, w, 0.0, nullptr, 0.0, nullptr, nullptr, len));
                for (int k = 0; k < it; ++k) {
                    const double a = H[(size_t)k * m + it], c = H[(size_t)(k + 1) * m + it];
                    H[(size_t)k * m + it] = cs[k] * a + sn[k] * c;
                    H[(size_t)(k + 1) * m + it] = -sn[k] * a + cs[k] * c;
                }
                const double denom = std::hypot(H[(size_t)it * m + it], H[(size_t)(it + 1) * m + it]);
                if (denom == 0.0) {
                    res.reason = CTL_DIVERGED_BREAKDOWN;
                    break;
                }
                cs[it] = H[(size_t)it * m + it] / denom;
                sn[it] = H[(size_t)(it + 1) * m + it] / denom;
                H[(size_t)it * m + it] = denom;
                H[(size_t)(it + 1) * m + it] = 0.0;
                g[it + 1] = -sn[it] * g[it];
                g[it] = cs[it] * g[it];
                rnorm = std::fabs(g[it + 1]);
                ++it;
                ++res.its;
                record(rnorm);
                res.reason = conv(rnorm);
                if (happy && res.reason == 0) res.reason = CTL_CONVERGED_HAPPY_BREAKDOWN;
            }
            if (res.its >= o.max_it && res.reason == 0) res.reason = CTL_DIVERGED_ITS;
            if (it > 0) {
                std::vector<double> y(it);
                for (int k = it - 1; k >= 0; --k) {
                    double s = g[k];
                    for (int j = k + 1; j < it; ++j) s -= H[(size_t)k * m + j] * y[j];
                    y[k] = s / H[(size_t)k * m + k];
                }
                CTL_TRY(vec_maxpy_host(h, x, flexible ? Z : V, it, y.data(), 1.0, len));
            }
        }
        return CTL_OK;
    }

    int minres(const double *b, double *x)
    {
        Scratch vecs[7];
        for (Scratch &s : vecs) CTL_TRY(pool.take(&s));
        double *r1 = vecs[0], *r2 = vecs[1], *y = vecs[2], *v = vecs[3], *w = vecs[4], *w1 = vecs[5], *w2 = vecs[6];
        CTL_TRY(prec(b, y));
        double bb = 0.0;
        CTL_TRY(dot(b, y, &bb));
        if (bb < 0.0) {
            res.reason = CTL_DIVERGED_INDEFINITE_PC;
            return CTL_OK;
        }
        res.ref_norm = std::sqrt(bb);
        const Conv conv(o.rtol, o.atol, o.divtol, res.ref_norm);
        CTL_TRY(op(x, r1));
        CTL_TRY(vec_lincomb(h, r1, 1.0, b, -1.0, r1, 0.0, nullptr, nullptr, len));
        CTL_TRY(prec(r1, y));
        double beta1 = 0.0;
        CTL_TRY(dot(r1, y, &beta1));
        if (beta1 < 0.0) {
            res.reason = CTL_DIVERGED_INDEFINITE_PC;
            return CTL_OK;
        }
        beta1 = std::sqrt(beta1);
        record(beta1);
        res.reason = conv(beta1);
        if (res.reason || beta1 == 0.0) {
            if (res.reason == 0) res.reason = CTL_CONVERGED_ATOL;
            return CTL_OK;
        }
        double oldb = 0.0, beta = beta1, dbar = 0.0, epsln = 0.0, phibar = beta1, cs = -1.0, sn = 0.0;
        CTL_TRY(vec_zero(h, w, len));
        CTL_TRY(vec_zero(h, w2, len));
        CTL_TRY(vec_copy(h, r2, r1, len));
        const double eps = std::numeric_limits<double>::epsilon();
        while (res.reason == 0 && res.its < o.max_it) {
            CTL_TRY(vec_lincomb(h, v, 1.0 / beta, y, 0.0, nullptr, 0.0, nullptr, nullptr, len));
            CTL_TRY(op(v, y));
            if (res.its >= 1) CTL_TRY(vec_lincomb(h, y, 1.0, y, -(beta / oldb), r1, 0.0, nullptr, nullptr, len));
            double alfa = 0.0;
            CTL_TRY(dot(v, y, &alfa));
            CTL_TRY(vec_lincomb(h, y, 1.0, y, -(alfa / beta), r2, 0.0, nullptr, nullptr, len));
            double *freed = r1;
            r1 = r2;
            r2 = y;
            y = freed;
            CTL_TRY(prec(r2, y));
            oldb = beta;
            CTL_TRY(dot(r2, y, &beta));
            if (beta < 0.0) {
                res.reason = CTL_DIVERGED_INDEFINITE_PC;
                break;
            }
            beta = std::sqrt(beta);
            const double oldeps = epsln;
            const double delta = cs * dbar + sn * alfa;
            const double gbar = sn * dbar - cs * alfa;
            epsln = sn * beta;
            dbar = -cs * beta;
            const double gamma = std::max(std::hypot(gbar, beta), eps);
            cs = gbar / gamma;
            sn = beta / gamma;
            const double phi = cs * phibar;
            phibar = sn * phibar;
            // w <- (v - oldeps w2_old - delta w_old) / gamma, written into the retired w1 buffer
            CTL_TRY(vec_lincomb(h, w1, 1.0 / gamma, v, -oldeps / gamma, w2, -delta / gamma, w, nullptr, len));
            double *neww = w1;
            w1 = w2;
            w2 = w;
            w = neww;
            CTL_TRY(vec_lincomb(h, x, 1.0, x, phi, w, 0.0, nullptr, nullptr, len));
            ++res.its;
            const double rnorm = std::fabs(phibar);
            record(rnorm);
            res.reason = conv(rnorm);
            if (beta == 0.0 && res.reason == 0) res.reason = CTL_CONVERGED_HAPPY_BREAKDOWN;
        }
        if (res.its >= o.max_it && res.reason == 0) res.reason = CTL_DIVERGED_ITS;
        return CTL_OK;
    }
};

// MultiBlockSystem.solve of K's system on internal-layout vectors (u: initial guess in, solution out), timed with
// device events: the whole solve into seconds_total, each operator / pc application into seconds_mult / seconds_pc
int krylov_solve(Solver &K, const double *b_in, double *u)
{
    ctl_handle_s *h = K.h;
    ctl_solve_result &res = K.res;
    K.ks.next_event = 0;
    K.ks.spans.clear();
    memset(&res, 0, sizeof(res));
    EventPair ev;
    CTL_TRY(ev.create(h));
    CTL_CUDA(cudaEventRecord(ev.begin, h->stream));
    int rc;
    {
        Scratch b;
        rc = K.pool.take(&b);
        // correct_soln / correct_rhs (preconditioner/preconditioner.py:658-704)
        if (rc == CTL_OK) rc = vec_copy(h, b, b_in, K.len);
        if (rc == CTL_OK) rc = K.project(b, nullptr);
        if (rc == CTL_OK) rc = K.project(u, nullptr);
        if (rc == CTL_OK) rc = (K.o.ksp_type == CTL_KSP_MINRES) ? K.minres(b, u) : K.gmres(b, u);
        if (rc == CTL_OK) rc = K.project(u, nullptr);                   // 761-766
        if (rc == CTL_OK) rc = ctl_comm_check(h);
    }
    cudaEventRecord(ev.end, h->stream);
    cudaEventSynchronize(ev.end);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ev.begin, ev.end);
    res.seconds_total = ms * 1e-3;
    for (auto &sp : K.ks.spans) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, K.ks.events[sp.first].begin, K.ks.events[sp.first].end) == cudaSuccess)
            (sp.second == 0 ? res.seconds_mult : res.seconds_pc) += t * 1e-3;
    }
    return rc;
}

}  // namespace
