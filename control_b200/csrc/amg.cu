// Aggregation-AMG V-cycle on the device (SURVEY.md row K9): the inner solver of the
// Schur-complement time sweeps, standing in for "preonly + hypre boomeramg, max_iter 2"
// (control/control.py:2056-2067 and the nine other sites).  The hierarchy is set up on
// the host once per distinct matrix (amg_setup.cpp); a cycle is a fixed sequence of
// SpMV-family kernels (sell.cu), so the time sweeps can be captured in a CUDA graph.
//
// Launches per V(nu, nu) cycle and level (the sweeps are bound by the number of dependent launches):
//   pre-smoothing    zero guess: the first TWO Chebyshev steps are one kernel (p1 = s D^-1 b is formed on the fly
//                    and never stored), so nu = 3 costs 2 launches; non-zero guess: nu launches
//   residual + restriction   two kernels (restricting b - A x in ONE kernel through a precomputed R A was measured:
//                    its rows are so long that the kernel costs more than the two it replaces, 30 us against 9 + 7)
//   coarse solve     dense inverse (one GEMV) below coarse_max rows
//   prolongation     one kernel, out of place (x' = x + P x_c) so that every kernel is idempotent: on several
//                    GPUs the boundary rows of a product are computed twice (halo.cuh)
//   post-smoothing   nu launches
// Multi-GPU: every level above `rep_min` rows per rank is distributed by rows; each kernel pushes the boundary
// rows of its output to the ranks that gather them and waits for its own ghosts (halo.cuh); the first level below
// the threshold receives its right-hand side through a replicating exchange (owners compute their rows, push them to
// everybody, one small kernel unpacks the arrivals) and everything below it runs redundantly on every rank.
#include "amg.cuh"

#include <cstdlib>
#include <stdexcept>

#include "cheb_coefficients.h"

int amg_build_distributed(ctl_handle_s *h, PcState *xs, const AmgParams &p,
                          const std::shared_ptr<SellPattern> &fine_pattern, AmgHierarchyDev &H);      // halo.cu

static int dev_alloc(ctl_handle_s *h, double **p, size_t n)
{
    CTL_CUDA(cudaMalloc((void **)p, std::max<size_t>(n, 1) * sizeof(double)));
    CTL_CUDA(cudaMemsetAsync(*p, 0, std::max<size_t>(n, 1) * sizeof(double), h->stream));
    return CTL_OK;
}

// work vectors of one level (after the matrices and dinv are in place): n rows of L.A.nc components each
int amg_level_vectors(ctl_handle_s *h, AmgLevelDev &L, int level)
{
    const size_t nv = (size_t)L.n * L.A.nc;
    CTL_TRY(dev_alloc(h, &L.r, nv));
    CTL_TRY(dev_alloc(h, &L.t0, nv));
    CTL_TRY(dev_alloc(h, &L.t1, nv));
    CTL_TRY(dev_alloc(h, &L.t2, nv));
    if (level > 0) {
        CTL_TRY(dev_alloc(h, &L.x, nv));
        CTL_TRY(dev_alloc(h, &L.b, nv));
    }
    return CTL_OK;
}

int64_t amg_cycle_bytes(const AmgHierarchyDev &H)
{
    // per cycle and level: 2 nu smoother products (2 nu - 1 on the zero-guess side) + residual, restriction,
    // prolongation; each product streams its matrix once plus the vectors it touches.  A block hierarchy (nc
    // components) streams each matrix once and every vector but the Jacobi diagonal nc times.
    const AmgParams &p = H.params;
    const int nl = (int)H.dev.size();
    const int64_t nc = H.nc;
    int64_t bytes = 0;
    for (int l = 0; l < nl; ++l) {
        const AmgLevelDev &L = H.dev[l];
        if (l + 1 < nl) {
            const int nu_l = (l == 0 && p.nu_fine > 0) ? p.nu_fine : p.nu;
            bytes += (L.A.bytes_per_pass + (8ll + 32ll * nc) * L.n) * (2 * nu_l);
            bytes += L.P.bytes_per_pass + L.R.bytes_per_pass + 32ll * nc * L.n;
        } else if (L.Ainv) {
            bytes += 8ll * L.n * L.n;
        } else {
            bytes += (L.A.bytes_per_pass + (8ll + 32ll * nc) * L.n) * p.nu;
        }
    }
    return bytes;
}

int amg_build(ctl_handle_s *h, const HostCSR &A0, const AmgParams &p,
              const std::shared_ptr<SellPattern> &fine_pattern, AmgHierarchyDev &H, PcState *xs)
{
    H.params = p;
    try {
        if (H.host.empty()) amg_setup_host(A0, p, H.host);      // else: set up earlier (pc.cu builds many in parallel)
    } catch (const std::exception &e) {
        ctl_set_error(h, e.what());
        return CTL_ERR_STATE;
    }
    const int nl = (int)H.host.size();
    H.dev.assign(nl, AmgLevelDev());
    CTL_CHECK(H.nc == 1 || h->cfg.world == 1, CTL_ERR_ARG, "amg_build: block hierarchies run on one GPU only");
    if (h->cfg.world > 1) {
        CTL_CHECK(nl > 1, CTL_ERR_ARG, "amg_build: the problem is too small for a multi-rank hierarchy (single level)");
        CTL_TRY(amg_build_distributed(h, xs, p, fine_pattern, H));
    } else {
        for (int l = 0; l < nl; ++l) {
            AmgLevelHost &Lh = H.host[l];
            AmgLevelDev &Ld = H.dev[l];
            Ld.n = Lh.A.n_rows;
            Ld.rho = Lh.rho;
            if (l == 0 && fine_pattern) CTL_TRY(sell_set_values(h, fine_pattern, Lh.A.values.data(), Ld.A));
            else CTL_TRY(sell_from_csr(h, Lh.A, Ld.A));
            Ld.A.nc = H.nc;
            CTL_TRY(ctl_upload(h, &Ld.dinv, Lh.dinv.data(), (size_t)Ld.n));      // one entry per row: shared by the components
            CTL_TRY(amg_level_vectors(h, Ld, l));
            if (l + 1 < nl) {
                CTL_TRY(sell_from_csr(h, Lh.P, Ld.P));
                CTL_TRY(sell_from_csr(h, Lh.R, Ld.R));
                Ld.P.nc = Ld.R.nc = H.nc;
            } else if (!Lh.Ainv.empty()) {
                CTL_TRY(dense_inverse_upload(h, Lh.Ainv, Ld.n, &Ld.Ainv, &Ld.Ainv_ld));
            } else if (Lh.coarse_inverse) {
                CTL_TRY(dense_inverse_device(h, Lh.A, Lh.coarse_shift, &Ld.Ainv, &Ld.Ainv_ld));
            }
        }
    }
    H.bytes_per_cycle = amg_cycle_bytes(H);
    if (p.acc_lo > 0.0) {
        const size_t nv = (size_t)H.dev[0].n * H.nc;
        CTL_TRY(dev_alloc(h, &H.acc_r, nv));
        CTL_TRY(dev_alloc(h, &H.acc_z, nv));
        CTL_TRY(dev_alloc(h, &H.acc_p, nv));
    }
    return CTL_OK;
}

void amg_free(AmgHierarchyDev &H)
{
    cudaFree(H.acc_r);
    cudaFree(H.acc_z);
    cudaFree(H.acc_p);
    H.acc_r = H.acc_z = H.acc_p = nullptr;
    for (AmgLevelDev &L : H.dev) {
        sell_free(L.A);
        sell_free(L.P);
        sell_free(L.R);
        cudaFree(L.dinv);
        cudaFree(L.x);
        cudaFree(L.b);
        cudaFree(L.r);
        cudaFree(L.t0);
        cudaFree(L.t1);
        cudaFree(L.t2);
        cudaFree(L.Ainv);
    }
    H.dev.clear();
    H.host.clear();
    H.spaces.clear();
}

// a level vector as a kernel gathers it: owned entries + the ghosts of the plan's last exchange
static GVec gathered(const AmgLevelDev &, HaloPlan *plan, const double *v, const SellMat &)
{
    if (!plan) return GVec(v);
    return GVec(v, halo_ll(plan), halo_idx1(plan));
}

// nu Chebyshev steps on D^-1 A over [lo rho, hi rho] (oracle/cheb.py::chebyshev).
//   x_in == nullptr: zero initial guess; otherwise p_0 = x_in (its boundary rows already pushed on L.px).
// The result lands in x_out, which may be x_in.  No kernel overwrites one of its inputs: intermediate iterates
// rotate through t0 / t1 / t2 (p_k in W[(k - 1) % 3]; the prolongation leaves p_0 in t2, first rewritten at k = 3,
// when p_0 is dead).  Every iterate that a later kernel gathers is pushed on L.px.
static int smooth(ctl_handle_s *h, const AmgParams &p, AmgLevelDev &L, int l, const GVec &b, const double *x_in, double *x_out)
{
    double scale;
    std::vector<double> om;
    const int nu = (l == 0 && p.nu_fine > 0) ? p.nu_fine : p.nu;
    cheb_coefficients(p.lo * L.rho, p.hi * L.rho, nu, &scale, om);
    double *W[3] = {L.t0, L.t1, L.t2};
    const bool zero = (x_in == nullptr);
    auto where = [&](int k) -> double * {
        if (k == nu) return x_out;
        return W[(k - 1) % 3];
    };
    if (zero && nu == 1) {
        const HaloPush push = halo_push(L.px);
        return vec_dinv_scale(h, L.dinv, b.x, x_out, scale, L.n, push, L.A.nc);
    }
    if (!zero && nu == 1 && x_in == x_out) {      // the one step would overwrite the vector it gathers
        CTL_CHECK(!L.px, CTL_ERR_STATE, "smooth: degree 1 in place is not available on several GPUs");
        CTL_TRY(sell_cheb_step(h, L.A, L.dinv, b.x, nullptr, GVec(x_in), L.t0, 0.0, 1.0, scale));
        return vec_copy_n(h, x_out, L.t0, L.n * L.A.nc);
    }
    int k0;      // first step that still has to be taken
    if (zero) {
        // p_2 = w p_1 + w s D^-1 (b - A p_1), p_1 = s D^-1 b formed on the fly
        const GVec dinv = L.px ? GVec(L.dinv, L.dinv + L.n) : GVec(L.dinv);
        const HaloPush push = halo_push(L.px);
        CTL_TRY(sell_cheb_first2(h, L.A, dinv, b, where(2), scale, om[0], push));
        k0 = 3;
    } else {
        // p_1 = x + s D^-1 (b - A x)
        const GVec cur = gathered(L, L.px, x_in, L.A);
        const HaloPush push = halo_push(L.px);
        CTL_TRY(sell_cheb_step(h, L.A, L.dinv, b.x, nullptr, cur, where(1), 0.0, 1.0, scale, 0.0, push));
        k0 = 2;
    }
    for (int k = k0; k <= nu; ++k) {
        const double w = om[k - 2];
        const GVec cur = gathered(L, L.px, where(k - 1), L.A);
        const HaloPush push = halo_push(L.px);
        if (zero && k == 3) {
            // p_{k-2} = p_1 was never stored: the kernel rebuilds it from b
            CTL_TRY(sell_cheb_step(h, L.A, L.dinv, b.x, nullptr, cur, where(k), 1.0 - w, w, w * scale, scale, push));
        } else {
            const double *prev = (k == 2) ? x_in : where(k - 2);
            CTL_TRY(sell_cheb_step(h, L.A, L.dinv, b.x, prev, cur, where(k), 1.0 - w, w, w * scale, 0.0, push));
        }
    }
    return CTL_OK;
}

// one V-cycle on level l: x <- cycle(b, x) (x_is_zero: x holds nothing yet).  b: the level's right-hand side with
// its ghosts (multi-GPU) as the kernels gather it.
static int vcycle(ctl_handle_s *h, AmgHierarchyDev &H, int l, const GVec &b, double *x, bool x_is_zero)
{
    AmgLevelDev &L = H.dev[l];
    const int last = (int)H.dev.size() - 1;
    if (l == last) {
        if (L.Ainv) return dense_gemv(h, L.Ainv, b.x, x, L.n, L.Ainv_ld, L.A.nc);
        return smooth(h, H.params, L, l, b, x_is_zero ? nullptr : x, x);
    }
    AmgLevelDev &C = H.dev[l + 1];
    CTL_TRY(smooth(h, H.params, L, l, b, x_is_zero ? nullptr : x, x));
    // right-hand side of the coarse level: the restricted residual.  Its producer pushes what the coarse level's
    // first kernels gather (distributed coarse level) or replicates it (first replicated level).
    HaloPush cpush;
    if (C.prep) cpush = halo_push(C.prep);
    else if (C.pb) cpush = halo_push(C.pb);
    double *cb = C.b;
    {
        // (the gathered vector is described BEFORE the next exchange of its plan is drawn: both read the plan's counter)
        HaloPlan *plan_r = L.pr ? L.pr : L.px;
        const GVec gx = gathered(L, L.px, x, L.A);
        const HaloPush push_r = halo_push(plan_r);
        CTL_TRY(sell_spmv(h, L.A, gx, L.r, b.x, SELL_RESIDUAL, push_r));
        const GVec gr = gathered(L, plan_r, L.r, L.R);
        CTL_TRY(sell_spmv(h, L.R, gr, cb, nullptr, SELL_ASSIGN, cpush));
    }
    GVec gcb(cb);
    if (C.prep) CTL_TRY(halo_unpack(h, C.prep, cb + C.prep->n_own));      // the other ranks' rows behind my own
    else if (C.pb) gcb = GVec(cb, halo_ll(C.pb), halo_idx1(C.pb));
    CTL_TRY(vcycle(h, H, l + 1, gcb, C.x, true));
    // x' = x + P x_c, out of place into t2; then the post-smoothing brings the result back into x
    const GVec gxc = gathered(C, C.px, C.x, L.P);
    const HaloPush push_x = halo_push(L.px);
    CTL_TRY(sell_spmv(h, L.P, gxc, L.t2, x, SELL_BPLUS, push_x));
    CTL_TRY(smooth(h, H.params, L, l, b, L.t2, x));
    return CTL_OK;
}

namespace {
// out = a x + b y + c z on n-vectors (x may be null when a == 0; out may alias x)
__global__ void lincomb3_kernel(double *out, double a, const double *x, double b, const double *__restrict__ y,
                                double c, const double *__restrict__ z, int n)
{
    pdl_sync();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double r = c * z[i];
    if (y) r = fma(b, y[i], r);
    if (x) r = fma(a, x[i], r);
    out[i] = r;
}
}  // namespace

int amg_solve(ctl_handle_s *h, AmgHierarchyDev &H, const double *b, double *x, bool b_exchanged)
{
    const AmgParams &p = H.params;
    AmgLevelDev &L0 = H.dev[0];
    if (L0.pb && !b_exchanged) CTL_TRY(halo_exchange_now(h, L0.pb, b));
    const GVec gb = L0.pb ? GVec(b, halo_ll(L0.pb), halo_idx1(L0.pb)) : GVec(b);
    if (p.acc_lo <= 0.0) {
        for (int c = 0; c < p.cycles; ++c) CTL_TRY(vcycle(h, H, 0, gb, x, c == 0));
        return CTL_OK;
    }
    // Chebyshev semi-iteration on (V-cycle * A) over [acc_lo, acc_hi]: oracle/amg.py::solve (one GPU only)
    CTL_CHECK(!L0.px, CTL_ERR_STATE, "amg_solve: accelerated cycles are not available on several GPUs");
    const int n = L0.n * H.nc;      // the vector work runs over every component
    double scale;
    std::vector<double> om;
    cheb_coefficients(p.acc_lo, p.acc_hi, p.cycles, &scale, om);
    double *buf[2] = {x, H.acc_p};
    auto slot = [&](int k) { return (p.cycles - k) & 1; };      // p_cycles lands in x
    const int blocks = ceil_div(n, 256);
    CTL_TRY(vcycle(h, H, 0, gb, H.acc_z, true));
    pdl_launch(h, blocks, 256, lincomb3_kernel, buf[slot(1)], 0.0, nullptr, 0.0, nullptr, scale, H.acc_z, n);
    h->launches++;
    for (int k = 2; k <= p.cycles; ++k) {
        const double w = om[k - 2];
        CTL_TRY(sell_spmv(h, L0.A, GVec(buf[slot(k - 1)]), H.acc_r, b, SELL_RESIDUAL));
        CTL_TRY(vcycle(h, H, 0, GVec(H.acc_r), H.acc_z, true));
        pdl_launch(h, blocks, 256, lincomb3_kernel, buf[slot(k)], 1.0 - w, k == 2 ? nullptr : buf[slot(k - 2)], w,
                                                      buf[slot(k - 1)], w * scale, H.acc_z, n);
        h->launches++;
    }
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}
