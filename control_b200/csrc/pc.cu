// In-built block preconditioner of Control.Instationary on the device
// (Instationary.construct_pc -> pc_linear, control/control.py:1943-2440), wrapped as
// Preconditioner.apply (preconditioner/preconditioner.py:562-656).
//
//   setup   once per matrix set: Jacobi diagonal of assemble(M, bcs); SELL copies of M and
//           of the sub/super-diagonal blocks of L_hat; one AMG hierarchy per DISTINCT
//           diagonal block (block_ii + shift M, assembled with bcs).  The reference
//           re-assembles and re-sets-up each of them at every time step of every
//           application (control/control.py:2056-2067 ...).
//   apply   (1,1) block: batched Chebyshev/Jacobi in the time-fastest layout
//           (pc_batched.cu); Schur block: right-hand side batched, then the forward and
//           backward time sweeps on time-slowest columns, one AMG solve per step.  The
//           sweeps are sequential in time as in the reference (control.py:2077, 2158) and
//           are replayed from ONE CUDA graph (about 70 small kernels per time step).
#include "pc.cuh"

#include <atomic>
#include <chrono>
#include <cstdio>
#include <map>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <thread>

#include "cheb_coefficients.h"
#include "vec_ops.cuh"

namespace {

// values of (w K_level(^T) + m_coef M) on the GLOBAL pattern, assembled with bcs when
// `identity`: constrained rows and columns zeroed, unit diagonal (Firedrake's
// assemble(a, bcs=...), control/control.py:2057-2059); otherwise rows and columns zeroed.
void combine_global(ctl_handle_s *h, int level, bool transposed, double w, double m_coef, bool identity,
                    std::vector<double> &out)
{
    const std::vector<int> &ip = h->h_indptr, &ix = h->h_indices;
    const int lv = h->h_K.size() > 1 ? level : 0;
    const std::vector<double> &Kv = h->h_K[lv];
    const std::vector<double> *KTv = h->h_KT.empty() ? nullptr : &h->h_KT[lv];
    out.assign(ix.size(), 0.0);
    for (int r = 0; r < h->n; ++r) {
        for (int k = ip[r]; k < ip[r + 1]; ++k) {
            const int c = ix[k];
            if (h->h_bcmask[r] || h->h_bcmask[c]) {
                out[k] = (identity && r == c) ? 1.0 : 0.0;
                continue;
            }
            double kv = 0.0;
            if (w != 0.0) {
                if (!transposed) kv = Kv[k];
                else if (KTv) kv = (*KTv)[k];
                else if (!h->h_tperm.empty()) kv = Kv[h->h_tperm[k]];
                else {
                    // entry (c, r) of the structurally symmetric pattern
                    const int *b = ix.data() + ip[c], *e = ix.data() + ip[c + 1];
                    const int *f = std::lower_bound(b, e, r);
                    kv = Kv[f - ix.data()];
                }
            }
            out[k] = w * kv + m_coef * h->h_M[k];
        }
    }
}

HostCSR global_csr(ctl_handle_s *h, const std::vector<double> &vals)
{
    HostCSR A;
    A.n_rows = A.n_cols = h->n;
    A.indptr = h->h_indptr;
    A.indices = h->h_indices;
    A.values = vals;
    return A;
}

// restrict global-pattern values to this rank's rows (local entry order)
std::vector<double> local_values(ctl_handle_s *h, const std::vector<double> &global_vals)
{
    std::vector<double> v(h->loc_entry.size());
    for (size_t p = 0; p < v.size(); ++p) v[p] = global_vals[h->loc_entry[p]];
    return v;
}

// ---- block-scalar sweeps (ctl_set_block_size): sweep matrices of the form I_bs (x) S on interleaved dofs,
// dof = bs node + comp, are set up and run as the scalar S on bs components
// The scalar pattern: the entries of the component-0 rows that lie in component-0 columns, numbered by node; src[p] is
// the global entry the scalar entry p is read from.
struct ScalarPattern {
    HostCSR A;                     // values unused
    std::vector<int64_t> src;
};

void scalar_pattern(const ctl_handle_s *h, int bs, ScalarPattern &out)
{
    const std::vector<int> &ip = h->h_indptr, &ix = h->h_indices;
    const int nn = h->n / bs;
    out.A.n_rows = out.A.n_cols = nn;
    out.A.indptr.assign(nn + 1, 0);
    out.A.indices.clear();
    out.src.clear();
    for (int i = 0; i < nn; ++i) {
        const int r = bs * i;
        for (int k = ip[r]; k < ip[r + 1]; ++k)
            if (ix[k] % bs == 0) {
                out.A.indices.push_back(ix[k] / bs);
                out.src.push_back(k);
            }
        out.A.indptr[i + 1] = (int)out.A.indices.size();
    }
}

std::vector<double> scalar_values(const ScalarPattern &sp, const std::vector<double> &global_vals)
{
    std::vector<double> v(sp.src.size());
    for (size_t p = 0; p < v.size(); ++p) v[p] = global_vals[sp.src[p]];
    return v;
}

HostCSR scalar_csr(const ScalarPattern &sp, const std::vector<double> &global_vals)
{
    HostCSR A = sp.A;
    A.values = scalar_values(sp, global_vals);
    return A;
}

// Values on the global pattern have the structure I_bs (x) S when no entry couples two components and the bs component
// blocks are equal entry for entry, bitwise; an absent entry and a stored zero both count as 0.  (A Dirichlet list that
// constrains only some components of a node breaks it: the constrained rows are identity rows.)
bool has_block_structure(const ctl_handle_s *h, int bs, const std::vector<double> &vals)
{
    const std::vector<int> &ip = h->h_indptr, &ix = h->h_indices;
    std::vector<std::pair<int, uint64_t>> first, other;
    for (int i = 0; i < h->n / bs; ++i) {
        for (int comp = 0; comp < bs; ++comp) {
            const int r = bs * i + comp;
            std::vector<std::pair<int, uint64_t>> &lst = comp == 0 ? first : other;
            lst.clear();
            for (int k = ip[r]; k < ip[r + 1]; ++k) {
                const double v = vals[k];
                if (v == 0.0) continue;
                if (ix[k] % bs != comp) return false;
                uint64_t bits;
                std::memcpy(&bits, &v, sizeof(bits));
                lst.emplace_back(ix[k] / bs, bits);
            }
            if (comp > 0 && other != first) return false;
        }
    }
    return true;
}

}  // namespace

void ctl_pc_free(ctl_handle_s *h)
{
    if (!h->pc) return;
    PcState &st = *h->pc;
    if (st.sweep_graph) cudaGraphExecDestroy(st.sweep_graph);
    for (auto &H : st.hier) amg_free(H);
    for (auto &m : st.off) sell_free(m);
    sell_free(st.Msell);
    cudaFree(st.d_mass_dinv);
    cudaFree(st.B);
    cudaFree(st.Uf);
    cudaFree(st.Ub);
    cudaFree(st.W);
    halo_arena_free(h, st.arena);
    h->pc.reset();
}

int ctl_pc_invalidate(ctl_handle_s *h)
{
    ctl_pc_free(h);
    return CTL_OK;
}

// a sweep vector with its ghosts behind the owned entries (multi-GPU: completed by halo_persist right after the
// solve that produced it, so later products need not wait)
static GVec ts_vec(const PcState &st, const double *v, int n_loc)
{
    if (!st.px0) return GVec(v);
    return GVec(v, v + n_loc);
}

static int enqueue_sweeps(ctl_handle_s *h, PcState &st)
{
    const int N = h->N, nl = h->n_loc;
    const size_t S = st.ts_stride;
    const bool cn = h->cfg.CN != 0;
    const double tau = h->cfg.tau, eps = h->cfg.epsilon;
    CTL_TRY(halo_epoch_begin(h));
    // forward sweep (control/control.py:2053-2116 CN, 2241-2328 BE).  The right-hand side of a step is formed out of
    // place (W = b_i -/+ Off u_{i-1}) by the kernel that also pushes its boundary rows to the neighbours.
    for (int i = 0; i < N; ++i) {
        const double *bi = st.B + i * S;
        if (i > 0) {
            const GVec up = ts_vec(st, st.Uf + (i - 1) * S, nl);
            const HaloPush push = halo_push(st.pb0);
            if (cn) CTL_TRY(sell_spmv(h, st.off[st.fwd_off[i]], up, st.W, bi, SELL_RESIDUAL, push));
            else CTL_TRY(sell_spmv(h, st.Msell, up, st.W, bi, SELL_BPLUS, push));     // b_i - (-M) u_{i-1}
            CTL_TRY(amg_solve(h, st.hier[st.fwd_h[i]], st.W, st.Uf + i * S, true));
        } else {
            CTL_TRY(amg_solve(h, st.hier[st.fwd_h[i]], bi, st.Uf + i * S, false));
        }
        CTL_TRY(halo_unpack(h, st.px0, st.Uf + i * S + nl));      // later products read its ghost entries
    }
    // middle scaling fused with the backward right-hand sides
    // (control/control.py:2118-2133 + 2158-2168 CN; 2330-2350 + 2375-2385 BE)
    for (int i = N - 1; i >= 0; --i) {
        double *bi = st.B + i * S;
        const GVec ui = ts_vec(st, st.Uf + i * S, nl);
        const GVec un = i + 1 < N ? ts_vec(st, st.Ub + (i + 1) * S, nl) : GVec();
        const HaloPush push = halo_push(st.pb0);
        if (cn) {
            // b_i = tau/2 M (T_2 u)_i - (L_hat^T)_{i,i+1} u_{i+1}; the block-diagonal variant has
            // no T_2 / T_2^-1 pair (oracle/pc.py::construct_pc_diagonal)
            const bool t2 = st.opts.mode == CTL_PCMODE_TRIANGULAR;
            const GVec up = (t2 && i > 0) ? ts_vec(st, st.Uf + (i - 1) * S, nl) : GVec();
            const SellMat &offm = un.x ? st.off[st.bwd_off[i]] : st.Msell;
            CTL_TRY(sell_spmv2(h, st.Msell, offm, ui, up, un, bi, 0.5 * tau, -1.0, push));
        } else {
            // b_i = tau M u_i (eps tau for the last block) - (-M) u_{i+1}
            const double a = (i == N - 1) ? eps * tau : tau;
            CTL_TRY(sell_spmv2(h, st.Msell, st.Msell, ui, GVec(), un, bi, a, 1.0, push));
        }
        CTL_TRY(amg_solve(h, st.hier[st.bwd_h[i]], bi, st.Ub + i * S, true));
        if (i > 0) CTL_TRY(halo_unpack(h, st.px0, st.Ub + i * S + nl));
    }
    return CTL_OK;
}

static int run_sweeps(ctl_handle_s *h, PcState &st)
{
    if (!st.sweep_graph) {
        const int64_t before = h->launches;
        cudaGraph_t graph = nullptr;
        CTL_CUDA(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeRelaxed));
        const int rc = enqueue_sweeps(h, st);
        const cudaError_t e = cudaStreamEndCapture(h->stream, &graph);
        if (rc != CTL_OK) {
            if (graph) cudaGraphDestroy(graph);
            return rc;
        }
        if (e != cudaSuccess) {
            ctl_set_error(h, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
            return CTL_ERR_CUDA;
        }
        CTL_CUDA(cudaGraphInstantiate(&st.sweep_graph, graph, 0));
        cudaGraphDestroy(graph);
        st.sweep_launches = h->launches - before;
        h->launches = before;
    }
    CTL_CUDA(cudaGraphLaunch(st.sweep_graph, h->stream));
    h->launches += st.sweep_launches;
    return CTL_OK;
}

// pc_fn(u_0, u_1, b_0, b_1) on time-fastest vectors.  wrap != 0 adds the nullspace handling
// of Preconditioner.apply: constrained entries of u take the values of b.
static int pc_fn_tf(ctl_handle_s *h, const double *b, double *u, bool wrap)
{
    CTL_CHECK(h->pc && h->pc->ready, CTL_ERR_STATE, "preconditioner: call ctl_pc_setup first");
    PcState &st = *h->pc;
    const size_t panel = (size_t)h->n_loc * h->ld;
    const double *b0 = b, *b1 = b + panel;
    double *u0 = u, *u1 = u + panel;
    const bool cn = h->cfg.CN != 0;
    const double tau = h->cfg.tau;
    Scratch s1, s2;
    CTL_TRY(h->pool.take(&s1));
    CTL_TRY(h->pool.take(&s2));
    double *btil = s1, *pa = s1 + panel, *pb = s2, *rhs = s2 + panel;
    // ---- (1,1) block: control/control.py:1997-2014 (CN), 2193-2206 (BE)
    const double *p_fin = nullptr;
    if (st.opts.solver_0 == CTL_S0_CHEBYSHEV) {
        double scale;
        std::vector<double> om;
        cheb_coefficients(st.opts.cheb_emin, st.opts.cheb_emax, st.opts.cheb_steps, &scale, om);
        double *buf[2] = {pa, pb};
        CTL_TRY(pcb_u0_first(h, b0, st.d_mass_dinv, btil, buf[1], scale));
        for (int k = 2; k <= st.opts.cheb_steps; ++k) {
            const double w = om[k - 2];
            if (h->n_halo > 0) CTL_TRY(ctl_halo_exchange_panel(h, buf[(k - 1) & 1]));
            CTL_TRY(pcb_cheb_step(h, st.d_mass_dinv, btil, k == 2 ? nullptr : buf[k & 1], buf[(k - 1) & 1], buf[k & 1],
                                  k == 2 ? 0.0 : 1.0 - w, w, w * scale));
        }
        p_fin = buf[st.opts.cheb_steps & 1];
    } else if (st.opts.solver_0 == CTL_S0_JACOBI) {
        CTL_TRY(pcb_u0_first(h, b0, st.d_mass_dinv, btil, pa, 1.0));
        p_fin = pa;
    } else {
        // Multigrid=True: AMG on assemble(M, bcs), column by column
        CTL_TRY(pcb_u0_first(h, b0, st.d_mass_dinv, btil, pa, 1.0));
        CTL_TRY(pcb_panel_to_ts(h, btil, st.B, st.ts_stride));
        CTL_TRY(halo_epoch_begin(h));
        for (int i = 0; i < h->N; ++i)
            CTL_TRY(amg_solve(h, st.hier[st.h_mass], st.B + i * st.ts_stride, st.Uf + i * st.ts_stride));
        CTL_TRY(pcb_ts_to_panel(h, st.Uf, pa, st.ts_stride));
        p_fin = pa;
    }
    const double sc = cn ? 2.0 / tau : 1.0 / tau;
    const double sc_last = cn ? sc : 1.0 / (tau * h->cfg.epsilon);
    CTL_TRY(pcb_u0_final(h, p_fin, wrap ? b0 : nullptr, u0, sc, sc_last));
    // ---- Schur block right-hand side: control/control.py:2016-2053 (CN), 2208-2237 (BE)
    if (st.opts.mode == CTL_PCMODE_TRIANGULAR) {
        // u0 has b's values on constrained rows when wrapping; the products must see
        // zeros there: the value arrays have constrained COLUMNS eliminated, so they do
        if (h->n_halo > 0) CTL_TRY(ctl_halo_exchange_panel(h, u0));
        CTL_TRY(pcb_schur_rhs(h, u0, b1, rhs));
    } else {
        CTL_TRY(pcb_schur_rhs(h, nullptr, b1, rhs));
    }
    CTL_TRY(pcb_panel_to_ts(h, rhs, st.B, st.ts_stride));
    // ---- forward / backward time sweeps
    CTL_TRY(run_sweeps(h, st));
    CTL_TRY(pcb_ts_to_panel(h, st.Ub, u1, st.ts_stride));
    return pcb_bc_fixup(h, h->d_bc_rows_all, h->n_bc_all, wrap ? b1 : nullptr, u1);
}

int ctl_pc_apply_tf(ctl_handle_s *h, const double *b_tf, double *u_tf) { return pc_fn_tf(h, b_tf, u_tf, true); }

static int pc_entry(ctl_handle_s *h, const double *b, double *u, int layout, bool wrap)
{
    CTL_CHECK(h && b && u, CTL_ERR_ARG, "ctl_pc_apply: null argument");
    CTL_CHECK(h->assembled, CTL_ERR_STATE, "ctl_pc_apply: ctl_assemble has not been called");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    if (layout == CTL_LAYOUT_TIME_FASTEST) {
        CTL_TRY(pc_fn_tf(h, b, u, wrap));
        return ctl_comm_check(h);
    }
    CTL_TRY(with_tf(h, layout, {b, nullptr}, u,
                    [&](const double *bt, double *ut) { return pc_fn_tf(h, bt, ut, wrap); }));
    return ctl_comm_check(h);
}

extern "C" {

int ctl_pc_default_options(ctl_pc_options *o)
{
    if (!o) return CTL_ERR_ARG;
    AmgParams d;
    o->mode = CTL_PCMODE_TRIANGULAR;
    o->solver_0 = CTL_S0_JACOBI;
    o->cheb_emin = 0.0;
    o->cheb_emax = 0.0;
    o->cheb_steps = 20;                  // "ksp_max_it": 20, control/control.py:1980
    o->amg_cycles = d.cycles;            // stands in for "pc_hypre_boomeramg_max_iter": 2, control.py:2065
    o->amg_nu = d.nu;
    o->amg_nu_fine = d.nu_fine;
    o->amg_max_levels = d.max_levels;
    o->amg_coarse_max = d.coarse_max;
    o->amg_theta = d.theta;
    o->amg_lo = d.lo;
    o->amg_hi = d.hi;
    o->amg_acc_lo = d.acc_lo;
    o->amg_acc_hi = d.acc_hi;
    return CTL_OK;
}

int ctl_amg_setup_probe(const int32_t *indptr, const int32_t *indices, const double *values, int32_t n,
                        const ctl_pc_options *opts, int32_t *n_levels, int32_t *level_n, int64_t *level_nnz,
                        double *level_rho, int32_t *aggregates)
{
    if (!indptr || !indices || !values || n <= 0 || !n_levels) return CTL_ERR_ARG;
    AmgParams p;
    if (opts) {
        p.theta = opts->amg_theta;
        p.max_levels = opts->amg_max_levels;
        p.coarse_max = opts->amg_coarse_max;
        p.nu = opts->amg_nu;
        p.nu_fine = opts->amg_nu_fine;
        p.lo = opts->amg_lo;
        p.hi = opts->amg_hi;
        p.cycles = opts->amg_cycles;
    }
    HostCSR A;
    A.n_rows = A.n_cols = n;
    A.indptr.assign(indptr, indptr + n + 1);
    A.indices.assign(indices, indices + indptr[n]);
    A.values.assign(values, values + indptr[n]);
    std::vector<AmgLevelHost> levels;
    try {
        amg_setup_host(A, p, levels);
    } catch (const std::exception &) {
        return CTL_ERR_STATE;
    }
    *n_levels = (int32_t)levels.size();
    for (size_t l = 0; l < levels.size() && l < 16; ++l) {
        if (level_n) level_n[l] = levels[l].A.n_rows;
        if (level_nnz) {             // entries that are not (numerically) zero: explicit zeros are a storage detail
            double amax = 0.0;
            for (double v : levels[l].A.values) amax = std::max(amax, std::fabs(v));
            int64_t cnt = 0;
            for (double v : levels[l].A.values) cnt += std::fabs(v) > 1e-13 * amax;
            level_nnz[l] = cnt;
        }
        if (level_rho) level_rho[l] = levels[l].rho;
    }
    if (aggregates && !levels[0].agg.empty()) std::copy(levels[0].agg.begin(), levels[0].agg.end(), aggregates);
    return CTL_OK;
}

namespace {
// CTL_SETUP_TIMING=1: where the time of ctl_pc_setup goes (stderr), next to the phases of the host AMG set-up
struct SetupLap {
    bool on = getenv("CTL_SETUP_TIMING") != nullptr;
    std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
    void operator()(const char *what)
    {
        if (!on) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[ctl pc_setup] %-28s %.3f s\n", what, std::chrono::duration<double>(now - t).count());
        t = now;
    }
};
}  // namespace

int ctl_pc_setup(ctl_handle h, const ctl_pc_options *opts)
{
    SetupLap lap;
    CTL_CHECK(h && opts, CTL_ERR_ARG, "ctl_pc_setup: null argument");
    CTL_CHECK(h->assembled, CTL_ERR_STATE, "ctl_pc_setup: ctl_assemble has not been called");
    CTL_CHECK(opts->mode == CTL_PCMODE_TRIANGULAR || opts->mode == CTL_PCMODE_DIAGONAL, CTL_ERR_ARG,
              "ctl_pc_setup: unknown mode");
    CTL_CHECK(opts->solver_0 >= CTL_S0_JACOBI && opts->solver_0 <= CTL_S0_AMG, CTL_ERR_ARG,
              "ctl_pc_setup: unknown solver_0");
    if (opts->solver_0 == CTL_S0_CHEBYSHEV)
        CTL_CHECK(opts->cheb_emax > opts->cheb_emin && opts->cheb_emin > 0 && opts->cheb_steps >= 1, CTL_ERR_ARG,
                  "ctl_pc_setup: Chebyshev needs 0 < e_min < e_max and at least one step");
    CTL_CHECK(opts->amg_cycles >= 1 && opts->amg_nu >= 1 && opts->amg_nu_fine >= 0 && opts->amg_max_levels >= 1,
              CTL_ERR_ARG, "ctl_pc_setup: bad AMG options");
    CTL_CHECK(opts->amg_acc_lo <= 0.0 || opts->amg_acc_hi > opts->amg_acc_lo, CTL_ERR_ARG,
              "ctl_pc_setup: AMG acceleration needs acc_lo < acc_hi");
    if (opts->mode == CTL_PCMODE_DIAGONAL)
        CTL_CHECK(h->cfg.CN && !h->per_level && h->k_symmetric, CTL_ERR_ARG,
                  "ctl_pc_setup: the block-diagonal (MINRES) variant needs CN and a time-independent symmetric K");
    CTL_CHECK(h->cfg.world == 1 || h->comm, CTL_ERR_STATE, "ctl_pc_setup: call ctl_comm_init first (world > 1)");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    ctl_pc_free(h);
    h->pc = std::make_shared<PcState>();
    PcState &st = *h->pc;
    st.opts = *opts;
    st.amg.theta = opts->amg_theta;
    st.amg.max_levels = opts->amg_max_levels;
    st.amg.coarse_max = opts->amg_coarse_max;
    st.amg.nu = opts->amg_nu;
    st.amg.nu_fine = opts->amg_nu_fine;
    st.amg.lo = opts->amg_lo;
    st.amg.hi = opts->amg_hi;
    st.amg.cycles = opts->amg_cycles;
    st.amg.acc_lo = opts->amg_acc_lo;
    st.amg.acc_hi = opts->amg_acc_hi;

    const int N = h->N, nl = h->n_loc, rb = h->row_begin;
    const bool cn = h->cfg.CN != 0;
    const double tau = h->cfg.tau, beta = h->cfg.beta, eps = h->cfg.epsilon;
    // transposed access into K without a stored K^T: one transposition map per pattern
    if (h->h_KT.empty() && !h->k_symmetric && h->h_tperm.size() != h->h_indices.size()) {
        const std::vector<int> &ip = h->h_indptr, &ix = h->h_indices;
        h->h_tperm.resize(ix.size());
        for (int r = 0; r < h->n; ++r)
            for (int k = ip[r]; k < ip[r + 1]; ++k) {
                const int c = ix[k];
                const int *b = ix.data() + ip[c], *e = ix.data() + ip[c + 1];
                h->h_tperm[k] = (int)(std::lower_bound(b, e, r) - ix.data());
            }
    }

    // Jacobi diagonal of assemble(M, bcs) and the list of constrained rows
    {
        std::vector<double> dinv(nl);
        for (int r = 0; r < nl; ++r) {
            const int g = rb + r;
            if (h->h_bcmask[g]) {
                dinv[r] = 1.0;
                continue;
            }
            double d = 0.0;
            for (int k = h->h_indptr[g]; k < h->h_indptr[g + 1]; ++k)
                if (h->h_indices[k] == g) d = h->h_M[k];
            CTL_CHECK(d != 0.0, CTL_ERR_ARG, "ctl_pc_setup: mass matrix has a zero diagonal entry");
            dinv[r] = 1.0 / d;
        }
        CTL_TRY(ctl_upload(h, &st.d_mass_dinv, dinv.data(), dinv.size()));
    }

    lap("transposition map, mass dinv");
    // multi-GPU: exchange geometry of everything that gathers through the mesh pattern, and the two level-0
    // exchange streams (iterates, right-hand sides) every hierarchy shares
    if (h->cfg.world > 1) {
        std::vector<int> part0(h->cfg.world + 1, 0);
        for (int r = 0; r < h->cfg.world; ++r) {
            const int base = h->n / h->cfg.world, rem = h->n % h->cfg.world;
            part0[r + 1] = part0[r] + base + (r < rem ? 1 : 0);
        }
        SpaceConsumer mesh;
        mesh.n_rows = h->n;
        mesh.indptr = h->h_indptr.data();
        mesh.indices = h->h_indices.data();
        mesh.row_part = part0.data();
        auto geom = std::make_shared<HaloGeom>();
        halo_geometry(h->cfg.world, h->cfg.rank, part0, {mesh}, false, *geom);
        CTL_TRY(halo_space_upload(h, geom, st.mesh_space));
        st.px0 = halo_arena_add(h, st.arena, st.mesh_space);
        st.pb0 = halo_arena_add(h, st.arena, st.mesh_space);
    }
    auto mesh_matrix = [&](SellMat &m) {
        if (h->cfg.world > 1) m.n_own = h->n_loc;
    };
    // distinct diagonal blocks -> AMG hierarchies; distinct off-diagonal blocks -> SELL
    const bool per_level = h->h_K.size() > 1;
    const bool sym = h->k_symmetric;
    std::map<std::tuple<int, int, double>, int> hier_index, off_index;
    // distinct diagonal blocks are only REGISTERED here; their hierarchies are set up afterwards, all
    // at once on the host threads (per-level K_i: 2N hierarchies per preconditioner setup)
    struct PendingHier { int level; bool transposed; double w, m_coef; };
    std::vector<PendingHier> pending;
    auto get_hier = [&](int level, bool transposed, double shift, double w, int *out) -> int {
        const auto key = std::make_tuple(per_level ? level : -1, (transposed && !sym) ? 1 : 0, shift);
        auto it = hier_index.find(key);
        if (it != hier_index.end()) {
            *out = it->second;
            return CTL_OK;
        }
        pending.push_back({level, transposed && !sym, w, 1.0 + shift});
        *out = hier_index[key] = (int)pending.size() - 1;
        return CTL_OK;
    };
    struct PendingOff { int level; bool transposed; double w, m_coef; };
    std::vector<PendingOff> pending_off;
    auto get_off = [&](int level, bool transposed, double w, double m_coef, int *out) -> int {
        const auto key = std::make_tuple(per_level ? level : -1, (transposed && !sym) ? 1 : 0, m_coef);
        auto it = off_index.find(key);
        if (it != off_index.end()) {
            *out = it->second;
            return CTL_OK;
        }
        pending_off.push_back({level, transposed && !sym, w, m_coef});
        *out = off_index[key] = (int)pending_off.size() - 1;
        return CTL_OK;
    };

    st.fwd_h.assign(N, -1);
    st.bwd_h.assign(N, -1);
    st.fwd_off.assign(N, -1);
    st.bwd_off.assign(N, -1);
    if (cn) {
        const double w = 0.5 * tau, c = 0.5 * tau / std::sqrt(beta);     // my_const, control.py:2051
        for (int i = 0; i < N; ++i) {
            // forward: block_10[(i,i)] + c M = w K_{i+1} + (1+c) M; block_10[(i,i-1)] + c M = w K_i + (c-1) M
            CTL_TRY(get_hier(i + 1, false, c, w, &st.fwd_h[i]));
            if (i > 0) CTL_TRY(get_off(i, false, w, c - 1.0, &st.fwd_off[i]));
            // backward: block_01[(i,i)] + c M = w K_i^T + (1+c) M; block_01[(i,i+1)] + c M = w K_{i+1}^T + (c-1) M
            CTL_TRY(get_hier(i, true, c, w, &st.bwd_h[i]));
            if (i + 1 < N) CTL_TRY(get_off(i + 1, true, w, c - 1.0, &st.bwd_off[i]));
        }
    } else {
        const double s = tau / std::sqrt(beta), se = std::sqrt(eps) * s;
        for (int i = 0; i < N; ++i) {
            const double sf = (i == 0) ? 0.0 : (i < N - 1 ? s : se);     // control.py:2243, 2279, 2312
            const double sb = (i == N - 1) ? se : (i > 0 ? s : 0.0);     // control.py:2358, 2391, 2422
            CTL_TRY(get_hier(i, false, sf, tau, &st.fwd_h[i]));
            CTL_TRY(get_hier(i, true, sb, tau, &st.bwd_h[i]));
        }
    }
    if (opts->solver_0 == CTL_S0_AMG) {
        pending.push_back({0, false, 0.0, 1.0});
        st.h_mass = (int)pending.size() - 1;
    }
    // block-scalar sweeps: only when EVERY sweep matrix (M, each distinct diagonal and off-diagonal block, the mass
    // hierarchy) has the structure I_bs (x) S; otherwise the whole handle takes the vector path.  Checked on the values
    // the set-up forms anyway, in parallel, before anything is built.
    st.bs = 1;
    if (h->block_size > 1) {
        const int bsz = h->block_size, nh = (int)pending.size(), n_off = (int)pending_off.size();
        const int n_tasks = 1 + nh + n_off;
        std::atomic<int> next{0};
        std::atomic<bool> ok{true};
        auto check = [&]() {
            std::vector<double> v;
            for (int i = next.fetch_add(1); i < n_tasks && ok.load(); i = next.fetch_add(1)) {
                if (i == 0) {
                    combine_global(h, 0, false, 0.0, 1.0, false, v);
                } else if (i <= nh) {
                    const PendingHier &q = pending[i - 1];
                    combine_global(h, q.level, q.transposed, q.w, q.m_coef, true, v);
                } else {
                    const PendingOff &o = pending_off[i - 1 - nh];
                    combine_global(h, o.level, o.transposed, o.w, o.m_coef, false, v);
                }
                if (!has_block_structure(h, bsz, v)) ok = false;
            }
        };
        int n_threads = std::max(1, setup_threads(std::max(1, (int)std::thread::hardware_concurrency())));
        n_threads = std::min(std::min(n_threads, n_tasks), 32);
        std::vector<std::thread> pool;
        for (int t = 1; t < n_threads; ++t) pool.emplace_back(check);
        check();
        for (auto &t : pool) t.join();
        if (ok) st.bs = bsz;
        lap("block structure check");
    }
    ScalarPattern spat;
    if (st.bs > 1) {
        // same depth as the vector hierarchy: the levels of S are half (a third) as large
        scalar_pattern(h, st.bs, spat);
        st.amg.coarse_max = (opts->amg_coarse_max + st.bs - 1) / st.bs;
        CTL_TRY(sell_build_pattern(h, spat.A, st.fine));
    } else {
        CTL_TRY(sell_build_pattern(h, h->loc, st.fine));
    }
    lap("fine SELL pattern");
    {
        std::vector<double> vals;
        combine_global(h, 0, false, 0.0, 1.0, false, vals);
        const std::vector<double> lv = st.bs > 1 ? scalar_values(spat, vals) : local_values(h, vals);
        CTL_TRY(sell_set_values(h, st.fine, lv.data(), st.Msell));
        st.Msell.nc = st.bs;
        mesh_matrix(st.Msell);
    }
    lap("mass matrix values");
    // host setup of all hierarchies in parallel, then the device uploads one after the other
    {
        const int nh = (int)pending.size(), n_off = (int)pending_off.size();
        st.hier.assign(nh, AmgHierarchyDev());
        std::vector<std::string> errors(nh);
        std::vector<std::vector<double>> off_values(n_off);
        // one process per GPU on one host: every rank sets the same hierarchies up, so each takes its share of the
        // cores (8 ranks x all 16 cores oversubscribed the box: 10-13 s of set-up at 8 GPUs against 2 s at one)
        int n_threads = setup_threads(std::max(1, (int)std::thread::hardware_concurrency() / std::max(1, h->cfg.world)));
        const int hw_threads = std::max(1, std::min(n_threads, 32));
        n_threads = std::max(1, std::min(std::min(n_threads, nh + n_off), 32));
        std::atomic<int> next{0};
        auto worker = [&]() {
            for (int i = next.fetch_add(1); i < nh + n_off; i = next.fetch_add(1)) {
                if (i >= nh) {                      // an off-diagonal block: values on the local pattern
                    const PendingOff &o = pending_off[i - nh];
                    std::vector<double> v;
                    combine_global(h, o.level, o.transposed, o.w, o.m_coef, false, v);
                    off_values[i - nh] = st.bs > 1 ? scalar_values(spat, v) : local_values(h, v);
                    continue;
                }
                try {
                    std::vector<double> v;
                    combine_global(h, pending[i].level, pending[i].transposed, pending[i].w, pending[i].m_coef, true, v);
                    // the workers share the host: each hierarchy gets its share of the threads
                    amg_setup_host(st.bs > 1 ? scalar_csr(spat, v) : global_csr(h, v), st.amg, st.hier[i].host,
                                   std::max(1, hw_threads / n_threads));
                } catch (const std::exception &e) {
                    errors[i] = e.what();
                }
            }
        };
        if (n_threads == 1) {
            worker();
        } else {
            std::vector<std::thread> pool;
            for (int t = 0; t < n_threads; ++t) pool.emplace_back(worker);
            for (auto &t : pool) t.join();
        }
        lap("host AMG set-up (all)");
        for (int i = 0; i < nh; ++i) {
            CTL_CHECK(errors[i].empty(), CTL_ERR_STATE, errors[i]);
            st.hier[i].nc = st.bs;
            CTL_TRY(amg_build(h, st.hier[i].host[0].A, st.amg, st.fine, st.hier[i]));
        }
        lap("formats, uploads, inverse");
        st.off.assign(n_off, SellMat());
        for (int i = 0; i < n_off; ++i) {
            CTL_TRY(sell_set_values(h, st.fine, off_values[i].data(), st.off[i]));
            st.off[i].nc = st.bs;
            mesh_matrix(st.off[i]);
            off_values[i] = std::vector<double>();
        }
        if (h->cfg.world > 1) CTL_TRY(halo_arena_finalize(h, st.arena));
        lap("off-diagonal blocks, arena");
    }

    st.ts_stride = (size_t)nl + h->n_halo;
    const size_t ts_bytes = (size_t)N * st.ts_stride * sizeof(double);
    CTL_CUDA(cudaMalloc((void **)&st.B, ts_bytes));
    CTL_CUDA(cudaMalloc((void **)&st.Uf, ts_bytes));
    CTL_CUDA(cudaMalloc((void **)&st.Ub, ts_bytes));
    CTL_CUDA(cudaMemsetAsync(st.B, 0, ts_bytes, h->stream));
    CTL_CUDA(cudaMemsetAsync(st.Uf, 0, ts_bytes, h->stream));
    CTL_CUDA(cudaMemsetAsync(st.Ub, 0, ts_bytes, h->stream));
    CTL_CUDA(cudaMalloc((void **)&st.W, st.ts_stride * sizeof(double)));
    CTL_CUDA(cudaMemsetAsync(st.W, 0, st.ts_stride * sizeof(double), h->stream));
    CTL_CUDA(cudaStreamSynchronize(h->stream));
    st.ready = true;
    return CTL_OK;
}

int ctl_pc_apply(ctl_handle h, const double *b, double *u, int layout) { return pc_entry(h, b, u, layout, true); }

int ctl_pc_fn(ctl_handle h, const double *b, double *u, int layout) { return pc_entry(h, b, u, layout, false); }

int ctl_set_pc_callback(ctl_handle h, ctl_pc_callback fn, void *user)
{
    CTL_CHECK(h, CTL_ERR_ARG, "ctl_set_pc_callback: null handle");
    h->pc_cb = fn;
    h->pc_cb_user = user;
    return CTL_OK;
}

// ---- AMG introspection
int32_t ctl_amg_num_hierarchies(ctl_handle h) { return (h && h->pc) ? (int32_t)h->pc->hier.size() : 0; }

int32_t ctl_amg_num_levels(ctl_handle h, int32_t hi)
{
    if (!h || !h->pc || hi < 0 || hi >= (int)h->pc->hier.size()) return 0;
    return (int32_t)h->pc->hier[hi].host.size();
}

#define AMG_LEVEL(h, hi, lvl)                                                                         \
    CTL_CHECK(h && h->pc && hi >= 0 && hi < (int)h->pc->hier.size() && lvl >= 0 &&                     \
                  lvl < (int)h->pc->hier[hi].host.size(),                                              \
              CTL_ERR_ARG, "AMG introspection: bad hierarchy / level");                                \
    const AmgLevelHost &L = h->pc->hier[hi].host[lvl]

int ctl_amg_level_size(ctl_handle h, int32_t hi, int32_t lvl, int32_t *n, int64_t *nnz_A, int64_t *nnz_P)
{
    AMG_LEVEL(h, hi, lvl);
    if (n) *n = L.A.n_rows;
    if (nnz_A) *nnz_A = L.A.nnz();
    if (nnz_P) *nnz_P = L.P.nnz();
    return CTL_OK;
}

int ctl_amg_get_csr(ctl_handle h, int32_t hi, int32_t lvl, int which, int32_t *indptr, int32_t *indices, double *values)
{
    AMG_LEVEL(h, hi, lvl);
    const HostCSR &A = which == 0 ? L.A : L.P;
    std::copy(A.indptr.begin(), A.indptr.end(), indptr);
    std::copy(A.indices.begin(), A.indices.end(), indices);
    std::copy(A.values.begin(), A.values.end(), values);
    return CTL_OK;
}

int ctl_amg_get_aggregates(ctl_handle h, int32_t hi, int32_t lvl, int32_t *agg)
{
    AMG_LEVEL(h, hi, lvl);
    std::copy(L.agg.begin(), L.agg.end(), agg);
    return CTL_OK;
}

int32_t ctl_pc_block_size(ctl_handle h) { return (h && h->pc && h->pc->ready) ? h->pc->bs : -1; }

int ctl_amg_solve(ctl_handle h, int32_t hi, const double *b, double *x)
{
    CTL_CHECK(h && h->pc && hi >= 0 && hi < (int)h->pc->hier.size() && b && x, CTL_ERR_ARG, "ctl_amg_solve: bad argument");
    CTL_CHECK(h->pc->hier[hi].nc != 2 || (((uintptr_t)b | (uintptr_t)x) & 15) == 0, CTL_ERR_ARG,
              "ctl_amg_solve: a block-size-2 hierarchy needs 16-byte aligned vectors");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    CTL_TRY(halo_epoch_begin(h));
    CTL_TRY(amg_solve(h, h->pc->hier[hi], b, x, false));
    return ctl_comm_check(h);
}

int ctl_time_amg(ctl_handle h, int32_t hi, int reps, int flush_l2, double *out)
{
    CTL_CHECK(h && h->pc && hi >= 0 && hi < (int)h->pc->hier.size() && out && reps > 0, CTL_ERR_ARG,
              "ctl_time_amg: bad argument");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    AmgHierarchyDev &H = h->pc->hier[hi];
    AmgLevelDev &L0 = H.dev[0];
    const int n = L0.n, nc = H.nc;
    const size_t nv = (size_t)n * nc + L0.n_ghost;      // ghost entries behind the owned ones (multi-GPU; left at zero)
    // Cold-cache timing of the two fine-level kernels: INPUTS LARGER THAN L2.  Each launch works on its own set of
    // vectors (dinv, b, p_prev, p_cur, out), and the sets rotate through more than twice the 126 MB of L2, so no
    // launch finds its operands there.  (Round 1 overwrote a 256 MB buffer between launches instead: that leaves
    // L2 full of DIRTY lines whose write-back then competes with the kernel's own traffic -- 18.4 us for the
    // stencil-format smoother against 12 us back to back -- and is no state the solve ever runs in.)
    constexpr int kSetVecs = 5;
    const size_t set_bytes = (size_t)kSetVecs * nv * sizeof(double);
    const int n_sets = flush_l2 ? (int)std::max<size_t>(2, ((size_t)300 << 20) / set_bytes + 1) : 1;
    DeviceArray<double> sets, flush;
    const size_t flush_bytes = 256u << 20;
    CTL_CUDA(sets.alloc((size_t)n_sets * kSetVecs * nv));
    CTL_CUDA(cudaMemset(sets, 0, (size_t)n_sets * set_bytes));
    if (flush_l2) CTL_CUDA(flush.alloc(flush_bytes / sizeof(double)));
    auto vec = [&](int set, int k) { return sets + ((size_t)set * kSetVecs + k) * nv; };      // k: 0 dinv 1 b 2 x 3 p 4 out
    {
        std::vector<double> hb((size_t)n * nc);
        for (size_t i = 0; i < hb.size(); ++i) hb[i] = std::sin(0.37 * i) + 0.1;
        for (int s = 0; s < n_sets; ++s) {      // (the Jacobi diagonal has one entry per row, whatever nc)
            CTL_CUDA(cudaMemcpy(vec(s, 0), L0.dinv, ((size_t)n + L0.n_ghost) * sizeof(double), cudaMemcpyDeviceToDevice));
            CTL_CUDA(cudaMemcpy(vec(s, 1), hb.data(), hb.size() * sizeof(double), cudaMemcpyHostToDevice));
            CTL_CUDA(cudaMemcpy(vec(s, 3), hb.data(), hb.size() * sizeof(double), cudaMemcpyHostToDevice));
        }
    }
    double *b = vec(0, 1), *x = vec(0, 2);
    EventPair ev;
    CTL_TRY(ev.create(h));
    // Each kernel is timed over `reps` launches between ONE pair of events: an event pair around a single 10 us
    // launch would add several microseconds of record / launch latency to it.  The whole inner solve (which = 2)
    // streams 2 GB per call; it is timed as (reps x [256 MB overwrite, solve]) minus (reps x [overwrite]).
    double acc[3] = {0, 0, 0};
    int64_t launches_solve = 0;
    int rc = CTL_OK;
    auto timed = [&](int which, bool with_kernel, float *ms) -> int {
        int r2 = which == 2 ? halo_epoch_begin(h) : CTL_OK;      // every rank times the same sequence
        cudaEventRecord(ev.begin, h->stream);
        for (int r = 0; r < reps && r2 == CTL_OK; ++r) {
            if (which == 2 && flush) cudaMemsetAsync(flush, r & 0xff, flush_bytes, h->stream);
            if (!with_kernel) continue;
            const int64_t l0 = h->launches;
            const int s = r % n_sets;
            const GVec gp = L0.px ? GVec(vec(s, 3), vec(s, 3) + (size_t)n * nc) : GVec(vec(s, 3));
            if (which == 0) r2 = sell_cheb_step(h, L0.A, vec(s, 0), vec(s, 1), vec(s, 2), gp, vec(s, 4), 0.3, 0.7, 0.1);
            else if (which == 1) r2 = sell_spmv(h, L0.A, gp, vec(s, 4), vec(s, 1), SELL_RESIDUAL);
            else r2 = amg_solve(h, H, b, x);
            launches_solve = h->launches - l0;
        }
        cudaEventRecord(ev.end, h->stream);
        cudaEventSynchronize(ev.end);
        cudaEventElapsedTime(ms, ev.begin, ev.end);
        return r2;
    };
    for (int which = 0; which < 3 && rc == CTL_OK; ++which) {
        float warm = 0.f, with_k = 0.f, without_k = 0.f;
        rc = timed(which, true, &warm);
        if (rc == CTL_OK) rc = timed(which, true, &with_k);
        if (rc == CTL_OK && which == 2) rc = timed(which, false, &without_k);
        acc[which] = with_k - ((flush && which == 2) ? without_k : 0.f);
    }
    const double mat = (double)L0.A.bytes_per_pass;      // matrix stream of the format in use (sell_format.h)
    out[0] = acc[0] / reps;
    out[1] = mat + (8.0 + 32.0 * nc) * n;    // matrix + dinv, b, p_prev, p_cur, out (the vectors nc times, dinv once)
    out[2] = acc[1] / reps;
    out[3] = mat + 24.0 * nc * n;            // matrix + b, x, r
    out[4] = acc[2] / reps;
    out[5] = (double)H.bytes_per_cycle * H.params.cycles;
    out[6] = (double)launches_solve;
    return rc;
}

}  // extern "C"
