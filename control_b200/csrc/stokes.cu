// Instationary Stokes control on the device: the outer system of
// Control.Instationary.incompressible_linear_solve (control/control.py:3592-4725), its operator
// (MultiBlockSystemMatrix.mult with sub_n_blocks = 2, preconditioner/preconditioner.py:375-543),
// the in-built pressure-Schur preconditioner (control/control.py:4299-4687) and the outer
// Krylov solve (4273-4297, 4688-4693).  Restated in oracle/stokes.py; this file follows it.
//
// Everything acting on the velocity blocks is the heat-type KKT machinery of the `velocity`
// handle (fused KKT apply, block preconditioner, inner GMRES).  What is new here:
//   panel_spmm     tau B / tau B^T on a whole [n x ld] time panel at once, with the sub-block
//                  T transform, the "- b_1", the 1/tau^2 scaling and the inverse transform of the
//                  Schur right-hand side folded into its epilogue (4363-4400)
//   colsum/shift   ConstantNullspace (preconditioner.py:133-155): per time block mean removal
//   K_p solves     AMG cycles per time block on the Neumann Laplacian (4300-4309)
//   M_p solves     batched Chebyshev/Jacobi on the pressure mass matrix (4311-4333)
// Outer vectors in the internal layout: [velocity time-fastest vector | pressure one].
//
// Several ranks: the velocity and the pressure rows are each split over the ranks by PETSc's rule (the two handles'
// own partitions).  Each rank keeps the rows of B for its pressure rows and the rows of B^T for its velocity rows;
// before a divergence product the rows of the other space that its rows read and other ranks own ("ghosts") arrive
// through NCCL (comm.cu: one exchange plan per product), and the ghost-aware product reads them from there.  The
// per-block means of ConstantNullspace and the norm of the Picard residual add the ranks' partial sums in one
// all-reduce; the K_p hierarchy is distributed like the sweep hierarchies, on an exchange state of its own.
#include <cmath>
#include <cstdlib>

#include "cheb_coefficients.h"
#include "comm.cuh"
#include "krylov.cuh"
#include "panel.cuh"

namespace {

struct DevCSR {
    int n_rows = 0, n_cols = 0;
    int n_own = 0;                // columns >= n_own are ghosts (several ranks)
    int *ptr = nullptr, *cols = nullptr;
    double *vals = nullptr;
};

enum { T_NONE = 0, T_ONE = 1, T_TWO = 2 };

}  // namespace

struct ctl_stokes_s {
    ctl_handle_s *hv = nullptr, *hp = nullptr;
    DevCSR B, BT;                 // B with the constrained velocity COLUMNS zeroed, and its transpose
    std::shared_ptr<LiftState> lift_div;   // the constrained columns of B before zeroing (ctl_stokes_lift_bc)
    ctl_stokes_pc_options opts{};
    bool pc_ready = false;
    std::shared_ptr<SellPattern> fine_p;
    AmgHierarchyDev Kp;
    bool have_Kp = false;
    std::vector<double> h_Kp_solver;   // ctl_stokes_set_laplacian_p: matrix of solver_K_p when it is not hp's K
    double *d_mp_dinv = nullptr;  // 1 / diag(M_p)
    double *ts_b = nullptr, *ts_x = nullptr;     // [2N][n_p] time-slowest columns of the K_p solves
    double *d_part = nullptr;     // partial column sums, [2 panels][blocks][ld]
    double *d_mean = nullptr;     // [2 sets][2 panels][ld]
    int colsum_blocks = 0;
    double *d_res_part = nullptr; // per-block partial norms of ctl_stokes_nonlinear_residual, then the norm
    int res_blocks = 0;
    ScratchPool pool;             // outer vectors (len() is never below the block-major length: ld >= N)
    KrylovState ks;
    ctl_pc_callback pc_cb = nullptr;   // user preconditioner P= of incompressible_linear_solve (control/control.py:4686-4689)
    void *pc_cb_user = nullptr;
    // several ranks
    ExchangePlan xB, xBT;         // ghosts of tau B X_v (velocity rows) and of tau B^T X_p (pressure rows)
    double *d_ghost_v = nullptr;  // [2 panels][xB.ghosts x ld]
    double *d_ghost_p = nullptr;  // [2 panels][xBT.ghosts x ld]
    std::unique_ptr<PcState> kp_x;   // exchange state (mesh geometry, level-0 plans, arena) of the K_p hierarchy
    int64_t len() const { return hv->vec_len() + hp->vec_len(); }
};

namespace {

constexpr int COLSUM_ROWS = 1024;   // rows per block of the column-sum kernel

// out[r, :] (+)= T_inv( post * ( T_fwd(alpha * (A X)[r, :]) - sub[r, :] ) ), columns >= N zeroed.
// HALO: columns >= n_own are ghost rows, read from the exchanged panel `ghost`.
template <int G, int CPL, bool HALO>
__device__ __forceinline__ void panel_spmm_rows(const int *__restrict__ ptr, const int *__restrict__ cols,
                                                const double *__restrict__ vals, const double *__restrict__ X,
                                                const double *__restrict__ ghost, int n_own,
                                                const double *__restrict__ sub, double *out, double alpha, double post,
                                                int t_fwd, int t_inv, int accumulate, int n_rows, int N, int ld)
{
    const RowMap m = row_map<G, CPL>(n_rows);
    const size_t off = (size_t)m.r * ld + m.c0;
    double acc[CPL];
#pragma unroll
    for (int q = 0; q < CPL; ++q) acc[q] = 0.0;
    const int kb = __ldg(ptr + m.r), ke = __ldg(ptr + m.r + 1);
#pragma unroll 2
    for (int k = kb; k < ke; ++k) {
        const int col = __ldg(cols + k);
        const double v = __ldg(vals + k);
        double x[CPL];
        if (HALO && col >= n_own) load_cols<CPL>(ghost + (size_t)(col - n_own) * ld + m.c0, x);
        else load_cols<CPL>(X + (size_t)col * ld + m.c0, x);
#pragma unroll
        for (int q = 0; q < CPL; ++q) acc[q] = fma(v, x[q], acc[q]);
    }
#pragma unroll
    for (int q = 0; q < CPL; ++q) acc[q] *= alpha;
    if (t_fwd != T_NONE) {
        double nb[CPL];
        if (t_fwd == T_ONE) time_next<G, CPL>(acc, nb, m.l);
        else time_prev<G, CPL>(acc, nb, m.l);
#pragma unroll
        for (int q = 0; q < CPL; ++q) acc[q] += nb[q];
    }
    if (sub) {
        double s[CPL];
        load_cols<CPL>(sub + off, s);
#pragma unroll
        for (int q = 0; q < CPL; ++q) acc[q] -= s[q];
    }
#pragma unroll
    for (int q = 0; q < CPL; ++q) {
        acc[q] *= post;
        if (m.c0 + q >= N) acc[q] = 0.0;
    }
    if (t_inv == T_ONE) t1_inv<G, CPL>(acc, m.l);
    else if (t_inv == T_TWO) t2_inv<G, CPL>(acc, m.l);
#pragma unroll
    for (int q = 0; q < CPL; ++q)
        if (m.c0 + q >= N) acc[q] = 0.0;
    if (!m.live) return;
    if (accumulate) {
#pragma unroll
        for (int q = 0; q < CPL / 2; ++q) {
            const double2 o = *reinterpret_cast<const double2 *>(out + off + 2 * q);
            acc[2 * q] += o.x;
            acc[2 * q + 1] += o.y;
        }
    }
    store_cols<CPL>(out + off, acc);
}

template <int G, int CPL>
__global__ void __launch_bounds__(256) panel_spmm_kernel(const int *__restrict__ ptr, const int *__restrict__ cols,
                                                        const double *__restrict__ vals, const double *__restrict__ X,
                                                        const double *__restrict__ sub, double *out, double alpha,
                                                        double post, int t_fwd, int t_inv, int accumulate, int n_rows,
                                                        int N, int ld)
{
    panel_spmm_rows<G, CPL, false>(ptr, cols, vals, X, nullptr, 0, sub, out, alpha, post, t_fwd, t_inv, accumulate,
                                   n_rows, N, ld);
}

template <int G, int CPL>
__global__ void __launch_bounds__(256) panel_spmm_halo_kernel(const int *__restrict__ ptr, const int *__restrict__ cols,
                                                             const double *__restrict__ vals, const double *__restrict__ X,
                                                             const double *__restrict__ ghost, int n_own,
                                                             const double *__restrict__ sub, double *out, double alpha,
                                                             double post, int t_fwd, int t_inv, int accumulate,
                                                             int n_rows, int N, int ld)
{
    panel_spmm_rows<G, CPL, true>(ptr, cols, vals, X, ghost, n_own, sub, out, alpha, post, t_fwd, t_inv, accumulate,
                                  n_rows, N, ld);
}

// in place: X[r, :] <- T_1^-1 / T_2^-1 X[r, :], columns >= N zeroed
template <int G, int CPL>
__global__ void __launch_bounds__(256) panel_tinv_kernel(double *X, int t_inv, int n_rows, int N, int ld)
{
    const RowMap m = row_map<G, CPL>(n_rows);
    const size_t off = (size_t)m.r * ld + m.c0;
    double v[CPL];
#pragma unroll
    for (int q = 0; q < CPL / 2; ++q) {
        const double2 o = *reinterpret_cast<const double2 *>(X + off + 2 * q);
        v[2 * q] = o.x;
        v[2 * q + 1] = o.y;
    }
    if (t_inv == T_ONE) t1_inv<G, CPL>(v, m.l);
    else t2_inv<G, CPL>(v, m.l);
#pragma unroll
    for (int q = 0; q < CPL; ++q)
        if (m.c0 + q >= N) v[q] = 0.0;
    if (!m.live) return;
    store_cols<CPL>(X + off, v);
}

// partial column sums of the two [n_rows x ld] panels of a pressure vector (blockIdx.y = panel);
// a fixed summation order keeps the result deterministic
__global__ void __launch_bounds__(256) colsum_partial_kernel(const double *__restrict__ X, double *__restrict__ part,
                                                            int n_rows, int ld, int rows_per_block)
{
    __shared__ double sh[256];
    X += (size_t)blockIdx.y * n_rows * ld;
    part += (size_t)blockIdx.y * gridDim.x * ld;
    const int c = threadIdx.x % ld, ro = threadIdx.x / ld, rs = blockDim.x / ld;
    const int r_end = min(n_rows, (int)(blockIdx.x + 1) * rows_per_block);
    double s = 0.0;
    for (int r = blockIdx.x * rows_per_block + ro; r < r_end; r += rs) s += X[(size_t)r * ld + c];
    sh[threadIdx.x] = s;
    __syncthreads();
    if (ro == 0) {
        for (int q = 1; q < rs; ++q) s += sh[q * ld + c];
        part[(size_t)blockIdx.x * ld + c] = s;
    }
}

// mean[panel][c] = sum_b part[panel][b][c] / n_rows   (one block per panel, ld threads; several ranks: n_rows = 1,
// the sums are all-reduced and then divided by mean_divide_kernel)
__global__ void colsum_finish_kernel(const double *__restrict__ part, double *__restrict__ mean, int blocks, int ld,
                                     int n_rows)
{
    const int c = threadIdx.x;
    part += (size_t)blockIdx.x * blocks * ld;
    double s = 0.0;
    for (int b = 0; b < blocks; ++b) s += part[(size_t)b * ld + c];
    mean[blockIdx.x * ld + c] = s / (double)n_rows;
}

// mean[i] /= n for i < count: the means from the all-reduced sums of several ranks
__global__ void mean_divide_kernel(double *mean, int count, double n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) mean[i] /= n;
}

// Epilogue of ctl_stokes_nonlinear_residual, one pass over the four panels of an internal-layout outer vector
// (rows [0, 2 n_v): velocity, then 2 n_p pressure rows):
//   velocity rows  R[r, :] <- b[r, :] - R[r, :], zero on constrained rows (R holds A_raw x there)
//   pressure rows  R already holds b_p - tau T(B x_v); read only
//   part[block]    sum over the block's rows of w ||T^-1 R[r, :]||^2, w = 1 (velocity) / w_p = 1 / tau^2 (pressure);
//                  T^-1 (CN only) is T_1^-1 on the first velocity and the second pressure panel, T_2^-1 on the other
//                  two -- the T each panel carries in stokes_apply_tf
// Every lane takes part in both scans so that rows of different panels may share a warp.
template <int G, int CPL>
__global__ void __launch_bounds__(256) stokes_residual_kernel(const double *__restrict__ b, double *R,
                                                             const uint8_t *__restrict__ bcmask,
                                                             double *__restrict__ part, int n_v, int n_p, int N,
                                                             int ld, int cn, double w_p)
{
    __shared__ double sh[8];
    const int n_rows = 2 * n_v + 2 * n_p;
    const RowMap m = row_map<G, CPL>(n_rows);
    const size_t off = (size_t)m.r * ld + m.c0;
    const bool vel = m.r < 2 * n_v;
    double v[CPL];
#pragma unroll
    for (int q = 0; q < CPL / 2; ++q) {
        const double2 o = *reinterpret_cast<const double2 *>(R + off + 2 * q);
        v[2 * q] = o.x;
        v[2 * q + 1] = o.y;
    }
    if (vel) {
        double s[CPL];
        load_cols<CPL>(b + off, s);
        const bool bc = bcmask[m.r < n_v ? m.r : m.r - n_v] != 0;
#pragma unroll
        for (int q = 0; q < CPL; ++q) v[q] = bc ? 0.0 : s[q] - v[q];
    }
#pragma unroll
    for (int q = 0; q < CPL; ++q)
        if (m.c0 + q >= N) v[q] = 0.0;
    if (vel && m.live) store_cols<CPL>(R + off, v);
    if (cn) {
        const bool one = vel ? m.r < n_v : m.r >= 2 * n_v + n_p;
        double a[CPL], c[CPL];
#pragma unroll
        for (int q = 0; q < CPL; ++q) a[q] = c[q] = v[q];
        t1_inv<G, CPL>(a, m.l);
        t2_inv<G, CPL>(c, m.l);
#pragma unroll
        for (int q = 0; q < CPL; ++q) v[q] = one ? a[q] : c[q];
    }
    double s = 0.0;
#pragma unroll
    for (int q = 0; q < CPL; ++q)
        if (m.c0 + q < N) s = fma(v[q], v[q], s);
    s = m.live ? (vel ? s : w_p * s) : 0.0;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_down_sync(0xffffffffu, s, d);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += sh[w];
        part[blockIdx.x] = t;
    }
}

// out = sqrt(sum_b part[b]) in a fixed order (one block of 256 threads); ROOT = false: the sum (several ranks add
// theirs before the root is taken)
template <bool ROOT>
__global__ void __launch_bounds__(256) residual_finish_kernel(const double *__restrict__ part, int blocks,
                                                              double *__restrict__ out)
{
    __shared__ double sh[256];
    double s = 0.0;
    for (int b = threadIdx.x; b < blocks; b += 256) s += part[b];
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = ROOT ? sqrt(sh[0]) : sh[0];
}

// out = v - mean_v (+ mean_w), both panels (2 * n_rows rows of ld columns)
__global__ void panel_shift_kernel(const double *v, double *out,
                                   const double *__restrict__ mean_v, const double *__restrict__ mean_w, int n_rows,
                                   int ld)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t panel = (size_t)n_rows * ld;
    if (i >= 2 * panel) return;
    const int p = i >= panel ? 1 : 0;
    const int c = (int)(i % ld);
    double s = mean_v[p * ld + c];
    if (mean_w) s -= mean_w[p * ld + c];
    out[i] = v[i] - s;
}

// out[r, :] = s * dinv[r] * in[r, :]
__global__ void panel_rowscale_kernel(const double *__restrict__ in, const double *__restrict__ dinv,
                                      double *__restrict__ out, double s, int n_rows, int ld)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)n_rows * ld) return;
    out[i] = s * dinv[i / ld] * in[i];
}

int upload_csr(ctl_handle_s *h, const HostCSR &A, int n_own, DevCSR &D)
{
    D.n_rows = A.n_rows;
    D.n_cols = A.n_cols;
    D.n_own = n_own;
    CTL_TRY(ctl_upload(h, &D.ptr, A.indptr.data(), A.indptr.size()));
    CTL_TRY(ctl_upload(h, &D.cols, A.indices.data(), A.indices.size()));
    CTL_TRY(ctl_upload(h, &D.vals, A.values.data(), A.values.size()));
    return CTL_OK;
}

void free_csr(DevCSR &D)
{
    cudaFree(D.ptr);
    cudaFree(D.cols);
    cudaFree(D.vals);
    D = DevCSR();
}

// ghost: the exchanged panel of the ghost rows of X (matrices with ghost columns only)
int panel_spmm(ctl_stokes_s *S, const DevCSR &A, const double *X, const double *ghost, const double *sub, double *out,
               double alpha, double post, int t_fwd, int t_inv, bool accumulate)
{
    ctl_handle_s *h = S->hv;
    const int ld = h->ld, nb = blocks_for(A.n_rows, ld);
    if (A.n_own < A.n_cols) {
        DISPATCH_G(ld, (panel_spmm_halo_kernel<GG, CC><<<nb, 256, 0, h->stream>>>(A.ptr, A.cols, A.vals, X, ghost, A.n_own,
                                                                            sub, out, alpha, post, t_fwd, t_inv,
                                                                            accumulate ? 1 : 0, A.n_rows, h->N, ld)));
    } else {
        DISPATCH_G(ld, (panel_spmm_kernel<GG, CC><<<nb, 256, 0, h->stream>>>(A.ptr, A.cols, A.vals, X, sub, out, alpha, post,
                                                                       t_fwd, t_inv, accumulate ? 1 : 0, A.n_rows, h->N,
                                                                       ld)));
    }
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

// several ranks: the ghost rows of `panels` input panels of a divergence product (B: velocity rows, B^T: pressure rows)
int div_exchange(ctl_stokes_s *S, bool transpose, const double *X, int panels)
{
    ctl_handle_s *h = S->hv;
    if (h->cfg.world == 1) return CTL_OK;
    const ExchangePlan &P = transpose ? S->xBT : S->xB;
    if (P.peers.empty()) return CTL_OK;
    const size_t panel = (size_t)(transpose ? S->hp->n_loc : h->n_loc) * h->ld;
    return exchange_plan_run(h, h->comm->comm, P, X, panel, panels, transpose ? S->d_ghost_p : S->d_ghost_v);
}

// The divergence blocks on both panels q of X, each with its sub-block transform (preconditioner.py:471-525, CN only):
//   B    (block_10): T_2 on panel 0, T_1 on panel 1     out[q] = T_inv(post (T(alpha B X[q]) - sub[q]))
//   B^T  (block_01): T_1 on panel 0, T_2 on panel 1     out[q] (+)= T(alpha B^T X[q])
// invert: T_inv = T (the Schur right-hand side of pc_fn), otherwise none.  X[q] are panels of the column space,
// out[q] and sub[q] panels of the row space.
int div_product(ctl_stokes_s *S, bool transpose, const double *X, const double *sub, double *out, double alpha,
                double post, bool invert, bool accumulate)
{
    ctl_handle_s *hv = S->hv, *hp = S->hp;
    const bool cn = hv->cfg.CN != 0;
    const size_t pv = (size_t)hv->n_loc * hv->ld, pp = (size_t)hp->n_loc * hp->ld;
    const size_t p_in = transpose ? pp : pv, p_out = transpose ? pv : pp;
    const DevCSR &A = transpose ? S->BT : S->B;
    const double *ghost = transpose ? S->d_ghost_p : S->d_ghost_v;
    const size_t g_panel = (transpose ? S->xBT : S->xB).ghosts.size() * hv->ld;
    CTL_TRY(div_exchange(S, transpose, X, 2));
    for (int q = 0; q < 2; ++q) {
        const int t = cn ? ((q == 0) == transpose ? T_ONE : T_TWO) : T_NONE;
        CTL_TRY(panel_spmm(S, A, X + q * p_in, ghost ? ghost + q * g_panel : nullptr, sub ? sub + q * p_out : nullptr,
                           out + q * p_out, alpha, post, t, invert ? t : T_NONE, accumulate));
    }
    return CTL_OK;
}

// in place on one time-fastest panel of handle h: X[r, :] <- T_1^-1 (which = 1) / T_2^-1 (which = 2) X[r, :]
int panel_tinv_h(ctl_handle_s *h, double *X, int which, int n_rows)
{
    const int ld = h->ld, nb = blocks_for(n_rows, ld);
    DISPATCH_G(ld, (panel_tinv_kernel<GG, CC><<<nb, 256, 0, h->stream>>>(X, which == 1 ? T_ONE : T_TWO, n_rows, h->N, ld)));
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

int panel_tinv(ctl_stokes_s *S, double *X, int t_inv, int n_rows) { return panel_tinv_h(S->hv, X, t_inv, n_rows); }

// ConstantNullspace on a pressure vector (both panels): out = v - mean(v) [+ mean(w)]
//   project / pre_mult_corrected_lhs / pc_pre_mult_corrected: w = null
//   post_mult_correct_lhs(x, y), pc_post_mult_correct(u, b):  w = x resp. b
// Several ranks: the per-rank column sums (of v, and of w) go through one all-reduce in rank order, then are divided by
// the global n_p, so every rank shifts by the same means and a run repeats bitwise for a given number of ranks.
int pressure_center(ctl_stokes_s *S, const double *v, const double *w, double *out)
{
    ctl_handle_s *h = S->hv;
    const bool several = h->cfg.world > 1;
    const int n_p = S->hp->n_loc, ld = h->ld, nb = S->colsum_blocks;
    const int div = several ? 1 : n_p;
    double *mean_v = S->d_mean, *mean_w = S->d_mean + 2 * ld;
    colsum_partial_kernel<<<dim3(nb, 2), 256, 0, h->stream>>>(v, S->d_part, n_p, ld, COLSUM_ROWS);
    colsum_finish_kernel<<<2, ld, 0, h->stream>>>(S->d_part, mean_v, nb, ld, div);
    h->launches += 2;
    if (w) {
        colsum_partial_kernel<<<dim3(nb, 2), 256, 0, h->stream>>>(w, S->d_part, n_p, ld, COLSUM_ROWS);
        colsum_finish_kernel<<<2, ld, 0, h->stream>>>(S->d_part, mean_w, nb, ld, div);
        h->launches += 2;
    }
    if (several) {
        const int count = (w ? 4 : 2) * ld;
        CTL_CUDA(cudaGetLastError());
        CTL_TRY(ctl_allreduce_sum(h, S->d_mean, count));
        mean_divide_kernel<<<ceil_div(count, 256), 256, 0, h->stream>>>(S->d_mean, count, (double)S->hp->n);
        h->launches++;
    }
    const size_t total = 2 * (size_t)n_p * ld;
    panel_shift_kernel<<<ceil_div(total, 256), 256, 0, h->stream>>>(v, out, mean_v, w ? mean_w : nullptr, n_p, ld);
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

// y = A x on the internal layout
int stokes_apply_tf(ctl_stokes_s *S, const double *x, double *y)
{
    ctl_handle_s *hv = S->hv, *hp = S->hp;
    const double tau = hv->cfg.tau;
    const double *x0 = x, *x1 = x + hv->vec_len();
    double *y0 = y, *y1 = y + hv->vec_len();
    CTL_TRY(ctl_kkt_apply_tf(hv, x0, y0));                       // block_00 (constrained rows: y = x)
    Scratch xc1;
    CTL_TRY(hp->pool.take(&xc1));
    CTL_TRY(pressure_center(S, x1, nullptr, xc1));               // pre_mult_corrected_lhs
    CTL_TRY(div_product(S, true, xc1, nullptr, y0, tau, 1.0, false, true));     // block_01 = diag(tau B^T)
    CTL_TRY(div_product(S, false, x0, nullptr, y1, tau, 1.0, false, false));    // block_10 = diag(tau B)
    return pressure_center(S, y1, x1, y1);                       // post_mult_correct_lhs
}

// solver_M_p on one panel: Chebyshev/Jacobi with fixed bounds or one Jacobi sweep
int mass_p_solve(ctl_stokes_s *S, const double *c, double *u, double *tmp)
{
    ctl_handle_s *hp = S->hp;
    ctl_handle_s *h = S->hv;
    const int n_p = hp->n_loc, ld = hp->ld;
    const size_t total = (size_t)n_p * ld;
    const int blocks = ceil_div(total, 256);
    if (S->opts.mass_p != CTL_S0_CHEBYSHEV) {
        panel_rowscale_kernel<<<blocks, 256, 0, h->stream>>>(c, S->d_mp_dinv, u, 1.0, n_p, ld);
        h->launches++;
        CTL_CUDA(cudaGetLastError());
        return CTL_OK;
    }
    const int steps = S->opts.mass_p_steps;
    double scale;
    std::vector<double> om;
    cheb_coefficients(S->opts.lambda_p_min, S->opts.lambda_p_max, steps, &scale, om);
    double *buf[2];
    buf[steps & 1] = u;             // iterate p_k lives in buf[k & 1]: p_steps lands in u
    buf[(steps & 1) ^ 1] = tmp;
    panel_rowscale_kernel<<<blocks, 256, 0, h->stream>>>(c, S->d_mp_dinv, buf[1], scale, n_p, ld);
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    for (int k = 2; k <= steps; ++k) {
        const double w = om[k - 2];
        if (hp->n_halo > 0) CTL_TRY(ctl_halo_exchange_panel(hp, buf[(k - 1) & 1]));
        CTL_TRY(pcb_cheb_step(hp, S->d_mp_dinv, c, k == 2 ? nullptr : buf[k & 1], buf[(k - 1) & 1], buf[k & 1],
                              k == 2 ? 0.0 : 1.0 - w, w, w * scale));
    }
    return CTL_OK;
}

// pc_fn(u_0, u_1, b_0, b_1) of control/control.py:4337-4513 (CN) / 4515-4687 (BE); wrap adds the
// nullspace handling of Preconditioner.apply (preconditioner/preconditioner.py:562-656)
int stokes_pc_run(ctl_stokes_s *S, const double *b, double *u, bool wrap)
{
    ctl_handle_s *hv = S->hv, *hp = S->hp;
    const bool cn = hv->cfg.CN != 0;
    const double tau = hv->cfg.tau;
    const int N = hv->N, n_p = hp->n_loc;
    const size_t pv = (size_t)hv->n_loc * hv->ld, pp = (size_t)n_p * hp->ld;
    const double *b0 = b, *b1 = b + hv->vec_len();
    double *u0 = u, *u1 = u + hv->vec_len();
    Scratch d1, s1, s2, s3;
    for (Scratch *s : {&d1, &s1, &s2, &s3}) CTL_TRY(hp->pool.take(s));
    const double *rhs1 = b1;
    if (wrap) {                                                 // pc_pre_mult_corrected
        CTL_TRY(pressure_center(S, b1, nullptr, d1));
        rhs1 = d1;
    }
    // ---- u_0: inner_its GMRES iterations on block_00 with the heat-type preconditioner, zero
    //      initial guess (4355-4361); the solve projects its right-hand side itself
    ctl_krylov_options io;
    ctl_krylov_default_options(&io);
    io.ksp_type = CTL_KSP_GMRES;
    io.max_it = S->opts.inner_its;
    io.rtol = 0.0;
    io.atol = 0.0;
    io.pc = CTL_PC_BUILTIN;
    ctl_solve_result ir;
    CTL_TRY(vec_zero(hv, u0, hv->vec_len()));
    CTL_TRY(ctl_solve_tf(hv, b0, u0, &io, &ir));
    // ---- u_1 = T^-1 ((T (tau B u_0) - b_1) / tau^2)
    CTL_TRY(div_product(S, false, u0, rhs1, s1, tau, 1.0 / (tau * tau), true, false));
    // ---- AMG cycles on K_p, one solve per time block
    for (int q = 0; q < 2; ++q) CTL_TRY(pcb_panel_to_ts(hp, s1 + q * pp, S->ts_b + (size_t)q * N * n_p, (size_t)n_p));
    CTL_TRY(halo_epoch_begin(hp));                              // several ranks: the K_p exchanges start a new epoch
    for (int j = 0; j < 2 * N; ++j) CTL_TRY(amg_solve(hp, S->Kp, S->ts_b + (size_t)j * n_p, S->ts_x + (size_t)j * n_p));
    for (int q = 0; q < 2; ++q) CTL_TRY(pcb_ts_to_panel(hp, S->ts_x + (size_t)q * N * n_p, s1 + q * pp, (size_t)n_p));
    // ---- multiply with the (untransformed) heat-type KKT blocks of the pressure space
    CTL_TRY(ctl_kkt_apply_tf(hp, s1, s2));
    if (cn) {
        CTL_TRY(panel_tinv(S, s2, T_ONE, n_p));
        CTL_TRY(panel_tinv(S, s2 + pp, T_TWO, n_p));
    }
    // ---- pressure mass solves
    for (int q = 0; q < 2; ++q) CTL_TRY(mass_p_solve(S, s2 + q * pp, u1 + q * pp, s3));
    if (wrap) {                                                 // pc_post_mult_correct
        CTL_TRY(pcb_bc_fixup(hv, hv->d_bc_rows_all, hv->n_bc_all, b0, u0));
        CTL_TRY(pcb_bc_fixup(hv, hv->d_bc_rows_all, hv->n_bc_all, b0 + pv, u0 + pv));
        CTL_TRY(pressure_center(S, u1, b1, u1));
    }
    return CTL_OK;
}

int stokes_pc_tf(ctl_stokes_s *S, const double *b, double *u, bool wrap)
{
    ctl_handle_s *h = S->hv;
    CTL_CHECK(S->pc_ready, CTL_ERR_STATE, "Stokes preconditioner: call ctl_stokes_pc_setup first");
    const int rc = stokes_pc_run(S, b, u, wrap);
    S->hv->launches += S->hp->launches;      // one counter for the whole system
    S->hp->launches = 0;
    return rc;
}

int outer_to_tf(ctl_stokes_s *S, const double *bm, double *tf)
{
    CTL_TRY(ctl_to_tf(S->hv, bm, tf));
    return ctl_to_tf(S->hp, bm + 2ll * S->hv->N * S->hv->n_loc, tf + S->hv->vec_len());
}

int outer_to_bm(ctl_stokes_s *S, const double *tf, double *bm)
{
    CTL_TRY(ctl_to_bm(S->hv, tf, bm));
    return ctl_to_bm(S->hp, tf + S->hv->vec_len(), bm + 2ll * S->hv->N * S->hv->n_loc);
}

struct StokesSolver : Solver {
    ctl_stokes_s *S;
    StokesSolver(ctl_stokes_s *S_, const ctl_krylov_options &o_, ctl_solve_result &r_)
        : Solver(S_->hv, o_, r_, S_->ks, S_->pool, S_->len(), "ctl_stokes_solve", S_->pc_cb, S_->pc_cb_user), S(S_) {}
    int apply_operator(const double *x, double *y) override { return stokes_apply_tf(S, x, y); }
    int apply_builtin_pc(const double *x, double *y) override { return stokes_pc_tf(S, x, y, true); }
    int to_bm(const double *tf, double *bm) override { return outer_to_bm(S, tf, bm); }
    int to_tf(const double *bm, double *tf) override { return outer_to_tf(S, bm, tf); }
    // velocity blocks: Dirichlet rows; pressure blocks: constants (full_nullspace_0 / _1, 3628-3652)
    int project(double *v, const double *wrap) override
    {
        CTL_TRY(Solver::project(v, wrap));
        double *v1 = v + S->hv->vec_len();
        return pressure_center(S, v1, wrap ? wrap + S->hv->vec_len() : nullptr, v1);
    }
};

// the K_p hierarchy and, on several ranks, its exchange arena (collective: every rank frees it at the same point)
void kp_free(ctl_stokes_s *S)
{
    if (S->kp_x) halo_arena_free(S->hp, S->kp_x->arena);
    S->kp_x.reset();
    if (S->have_Kp) amg_free(S->Kp);
    S->have_Kp = false;
}

// has a bounded wait of either handle's device-initiated exchange given up (ctl_comm_check)?  Both report through the
// velocity handle.
int stokes_comm_check(ctl_stokes_s *S)
{
    ctl_handle_s *h = S->hv;
    CTL_TRY(ctl_comm_check(h));
    const int rc = ctl_comm_check(S->hp);
    if (rc != CTL_OK) ctl_set_error(h, "pressure handle: " + S->hp->err);
    return rc;
}

// with_internal for the Stokes system: the caller's vectors are block-major
template <size_t K, class F>
int with_tf(ctl_stokes_s *S, const double *const (&in)[K], double *out, F fn)
{
    ctl_handle_s *h = S->hv;
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    return with_internal(
        S->pool, in, out, [S](const double *bm, double *tf) { return outer_to_tf(S, bm, tf); },
        [S](const double *tf, double *bm) { return outer_to_bm(S, tf, bm); }, fn);
}

}  // namespace

int ctl_panel_tinv(ctl_handle_s *h, double *X, int which, int n_rows) { return panel_tinv_h(h, X, which, n_rows); }

extern "C" {

int ctl_stokes_create(ctl_handle velocity, ctl_handle pressure, const int32_t *B_indptr, const int32_t *B_indices,
                      const double *B_values, ctl_stokes *out)
{
    ctl_handle_s *h = velocity;
    if (!h) return CTL_ERR_ARG;
    CTL_CHECK(pressure && B_indptr && B_indices && B_values && out, CTL_ERR_ARG, "ctl_stokes_create: null argument");
    CTL_CHECK(velocity->assembled && pressure->assembled, CTL_ERR_STATE,
              "ctl_stokes_create: assemble the velocity and pressure handles first");
    const ctl_config &a = velocity->cfg, &b = pressure->cfg;
    CTL_CHECK(a.n_t == b.n_t && a.CN == b.CN && a.tau == b.tau && a.beta == b.beta && a.device == b.device &&
                  a.rank == b.rank && a.world == b.world && velocity->stream == pressure->stream,
              CTL_ERR_ARG, "ctl_stokes_create: the two handles must share n_t, CN, tau, beta, rank, world, device and stream");
    CTL_CHECK(a.world == 1 || (velocity->comm && pressure->comm), CTL_ERR_STATE,
              "ctl_stokes_create: call ctl_comm_init on both handles first (world > 1)");
    CTL_CHECK(pressure->h_bc.empty(), CTL_ERR_ARG, "ctl_stokes_create: the pressure handle must not carry Dirichlet dofs");
    CTL_CUDA(cudaSetDevice(a.device));
    const int n_v = velocity->n, n_p = pressure->n;
    HostCSR B;
    B.n_rows = n_p;
    B.n_cols = n_v;
    B.indptr.assign(B_indptr, B_indptr + n_p + 1);
    const int64_t nnz = B.indptr[n_p];
    B.indices.assign(B_indices, B_indices + nnz);
    B.values.assign(B_values, B_values + nnz);
    for (int64_t k = 0; k < nnz; ++k)
        CTL_CHECK(B.indices[k] >= 0 && B.indices[k] < n_v, CTL_ERR_ARG, "ctl_stokes_create: column index out of range");
    std::shared_ptr<LiftState> lift_div;       // kept for the lifting of inhomogeneous velocity data
    CTL_TRY(ctl_lift_div_setup(velocity, B_indptr, B_indices, B_values, pressure->row_begin, pressure->n_loc, &lift_div));
    for (int64_t k = 0; k < nnz; ++k)
        if (velocity->h_bcmask[B.indices[k]]) B.values[k] = 0.0;      // the operator sees x with bcs zeroed
    HostCSR BT;
    csr_transpose(B, BT);
    ctl_stokes_s *S = new ctl_stokes_s();
    S->hv = velocity;
    S->hp = pressure;
    S->pool.init(h, S->len());
    S->lift_div = lift_div;
    int rc = CTL_OK;
    if (a.world == 1) {
        rc = upload_csr(h, B, n_v, S->B);
        if (rc == CTL_OK) rc = upload_csr(h, BT, n_p, S->BT);
    } else {
        // this rank's rows of B (pressure) and of B^T (velocity), each over the other space's split
        const int vb = velocity->row_begin, nv = velocity->n_loc, pb = pressure->row_begin, np = pressure->n_loc;
        rc = exchange_plan_build(h, B.indptr.data(), B.indices.data(), n_p, n_v, a.world, a.rank, S->xB);
        if (rc == CTL_OK) rc = exchange_plan_build(h, BT.indptr.data(), BT.indices.data(), n_v, n_p, a.world, a.rank, S->xBT);
        if (rc == CTL_OK) rc = upload_csr(h, local_rows(B, pb, np, vb, nv, S->xB.ghosts), nv, S->B);
        if (rc == CTL_OK) rc = upload_csr(h, local_rows(BT, vb, nv, pb, np, S->xBT.ghosts), np, S->BT);
        const size_t gv = 2 * S->xB.ghosts.size() * h->ld, gp = 2 * S->xBT.ghosts.size() * h->ld;
        if (rc == CTL_OK && gv && cudaMalloc((void **)&S->d_ghost_v, gv * sizeof(double)) != cudaSuccess) rc = CTL_ERR_CUDA;
        if (rc == CTL_OK && gp && cudaMalloc((void **)&S->d_ghost_p, gp * sizeof(double)) != cudaSuccess) rc = CTL_ERR_CUDA;
    }
    S->colsum_blocks = ceil_div(pressure->n_loc, COLSUM_ROWS);
    if (rc == CTL_OK && cudaMalloc((void **)&S->d_part, sizeof(double) * 2 * S->colsum_blocks * h->ld) != cudaSuccess) rc = CTL_ERR_CUDA;
    if (rc == CTL_OK && cudaMalloc((void **)&S->d_mean, sizeof(double) * 4 * h->ld) != cudaSuccess) rc = CTL_ERR_CUDA;
    S->res_blocks = blocks_for(2 * (velocity->n_loc + pressure->n_loc), h->ld);
    if (rc == CTL_OK && cudaMalloc((void **)&S->d_res_part, sizeof(double) * (S->res_blocks + 1)) != cudaSuccess)
        rc = CTL_ERR_CUDA;
    if (rc != CTL_OK) {
        if (h->err.empty()) ctl_set_error(h, "ctl_stokes_create: device allocation failed");
        ctl_stokes_destroy(S);
        return rc;
    }
    *out = S;
    return CTL_OK;
}

int ctl_stokes_destroy(ctl_stokes S)
{
    if (!S) return CTL_OK;
    cudaSetDevice(S->hv->cfg.device);
    cudaStreamSynchronize(S->hv->stream);
    free_csr(S->B);
    free_csr(S->BT);
    kp_free(S);
    cudaFree(S->d_ghost_v);
    cudaFree(S->d_ghost_p);
    cudaFree(S->d_mp_dinv);
    cudaFree(S->ts_b);
    cudaFree(S->ts_x);
    cudaFree(S->d_part);
    cudaFree(S->d_mean);
    cudaFree(S->d_res_part);
    delete S;
    return CTL_OK;
}

int ctl_stokes_lift_bc(ctl_stokes S, const double *g, double *b)
{
    if (!S) return CTL_ERR_ARG;
    ctl_handle_s *h = S->hv;
    CTL_CHECK(h->assembled, CTL_ERR_STATE, "ctl_stokes_lift_bc: the velocity handle is not assembled");
    if (h->h_bc.empty()) return CTL_OK;
    CTL_CHECK(g && b, CTL_ERR_ARG, "ctl_stokes_lift_bc: null g or b (the velocity handle has Dirichlet dofs)");
    CTL_TRY(ctl_lift_bc(h, g, b, CTL_LAYOUT_BLOCK_MAJOR));              // velocity rows: [2N blocks of n_v]
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    CTL_TRY(ctl_lift_div_apply(h, S->lift_div.get(), g, b + 2 * (size_t)h->N * h->n_loc, S->hp->n_loc));   // b_1_0
    return stokes_comm_check(S);
}

// Residual of the Navier-Stokes Picard loop (res_eval, control/control.py:4979-5072) on device vectors.  The
// reference takes it with the RAW coupling products (r00 -= tau B^T mu, r01 -= tau B^T p, r10 = -B v, r11 = -B zeta),
// so this is b - A_raw x: the operator of stokes_apply_tf without the ConstantNullspace corrections of the pressure
// parts, which would shift the residual by the per-block means of mu and p.  Norm: that of the untransformed,
// unscaled parts, ||T^-1 r_v||^2 + ||T^-1 r_p||^2 / tau^2.
int ctl_stokes_nonlinear_residual(ctl_stokes S, const double *b, const double *x, double *r, double *norm_host)
{
    if (!S) return CTL_ERR_ARG;
    ctl_handle_s *h = S->hv, *hp = S->hp;
    CTL_CHECK(b && x && r && norm_host, CTL_ERR_ARG, "ctl_stokes_nonlinear_residual: null argument");
    CTL_CHECK(r != b && r != x, CTL_ERR_ARG, "ctl_stokes_nonlinear_residual: r must not alias b or x");
    CTL_CHECK(h->assembled && hp->assembled, CTL_ERR_STATE,
              "ctl_stokes_nonlinear_residual: the velocity and pressure handles are not assembled");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    const bool cn = h->cfg.CN != 0, several = h->cfg.world > 1;
    const double tau = h->cfg.tau;
    const int n_v = h->n_loc, n_p = hp->n_loc, ld = h->ld;
    const int64_t lv = h->vec_len();
    double *partials = nullptr, *scalars = nullptr;
    CTL_TRY(vec_workspace(h, &partials, &scalars));                             // pinned staging of vec_read_scalars
    CTL_TRY(with_tf(S, {b, x, nullptr}, r, [&](const double *bt, const double *xt, double *yt) -> int {
        CTL_TRY(ctl_kkt_apply_tf(h, xt, yt));                                    // block_00 with D_v at the iterate
        CTL_TRY(div_product(S, true, xt + lv, nullptr, yt, tau, 1.0, false, true));         // + tau T(B^T x_p), raw x_p
        CTL_TRY(div_product(S, false, xt, bt + lv, yt + lv, tau, -1.0, false, false));      // r_p = b_p - tau T(B x_v)
        DISPATCH_G(ld, (stokes_residual_kernel<GG, CC><<<S->res_blocks, 256, 0, h->stream>>>(
                           bt, yt, h->d_bcmask, S->d_res_part, n_v, n_p, h->N, ld, cn ? 1 : 0, 1.0 / (tau * tau))));
        if (several)
            residual_finish_kernel<false><<<1, 256, 0, h->stream>>>(S->d_res_part, S->res_blocks, S->d_res_part + S->res_blocks);
        else
            residual_finish_kernel<true><<<1, 256, 0, h->stream>>>(S->d_res_part, S->res_blocks, S->d_res_part + S->res_blocks);
        h->launches += 2;
        CTL_CHECK(cudaGetLastError() == cudaSuccess, CTL_ERR_CUDA,
                  "ctl_stokes_nonlinear_residual: kernel launch failed");
        // several ranks: the sum of the squares over all rows, then the root of the same sum on every rank
        if (several) CTL_TRY(ctl_allreduce_sum(h, S->d_res_part + S->res_blocks, 1));
        return CTL_OK;
    }));
    CTL_TRY(vec_read_scalars(h, S->d_res_part + S->res_blocks, 1, norm_host));
    if (several) *norm_host = std::sqrt(*norm_host);
    return stokes_comm_check(S);
}

int64_t ctl_stokes_vec_len(ctl_stokes S) { return S ? 2ll * S->hv->N * ((int64_t)S->hv->n_loc + S->hp->n_loc) : 0; }

int ctl_stokes_pc_default_options(ctl_stokes_pc_options *o)
{
    if (!o) return CTL_ERR_ARG;
    ctl_pc_default_options(&o->velocity);
    // the aggregation hierarchy of the vector-P2 velocity operator contracts more slowly than the P1
    // one (energy norm, per V(3,3) cycle: 0.28 at 64^2, 0.34 at 128^2, worse at 512^2), and the inner
    // GMRES runs a fixed five iterations: at config C4 three cycles need > 100 outer iterations,
    // six need 18 (51.7 s against > 150 s)
    o->velocity.amg_cycles = 6;
    AmgParams d;
    o->inner_its = 5;                   // control/control.py:4358
    o->mass_p = CTL_S0_JACOBI;
    o->mass_p_steps = 20;               // control/control.py:4320
    o->lambda_p_min = o->lambda_p_max = 0.0;
    o->amg_p_nu = d.nu;
    o->amg_p_max_levels = d.max_levels;
    o->amg_p_coarse_max = d.coarse_max;
    // The reference: ONE BoomerAMG cycle (4300-4309).  The outer iteration count is very sensitive
    // to the accuracy of this solve (oracle measurements at 64^2: 25 / 20 / 15 / 10 outer iterations
    // with 1 / 2 / 4 / 6 cycles of this AMG, 10 with exact solves) while its cost is negligible next
    // to the velocity sweeps, so the stand-in runs six cycles.
    o->amg_p_cycles = 6;
    o->amg_p_theta = d.theta;
    o->amg_p_lo = d.lo;
    o->amg_p_hi = d.hi;
    return CTL_OK;
}

int ctl_stokes_set_laplacian_p(ctl_stokes S, const double *values_host)
{
    if (!S) return CTL_ERR_ARG;
    if (values_host)
        S->h_Kp_solver.assign(values_host, values_host + S->hp->h_indices.size());
    else
        S->h_Kp_solver.clear();
    S->pc_ready = false;
    return CTL_OK;
}

int ctl_stokes_pc_setup(ctl_stokes S, const ctl_stokes_pc_options *opts)
{
    if (!S) return CTL_ERR_ARG;
    ctl_handle_s *h = S->hv, *hp = S->hp;
    CTL_CHECK(opts, CTL_ERR_ARG, "ctl_stokes_pc_setup: null options");
    CTL_CHECK(opts->inner_its >= 1, CTL_ERR_ARG, "ctl_stokes_pc_setup: inner_its must be positive");
    CTL_CHECK(opts->mass_p == CTL_S0_JACOBI || opts->mass_p == CTL_S0_CHEBYSHEV, CTL_ERR_ARG,
              "ctl_stokes_pc_setup: mass_p must be Jacobi or Chebyshev");
    if (opts->mass_p == CTL_S0_CHEBYSHEV)
        CTL_CHECK(opts->lambda_p_max > opts->lambda_p_min && opts->lambda_p_min > 0 && opts->mass_p_steps >= 1, CTL_ERR_ARG,
                  "ctl_stokes_pc_setup: Chebyshev needs 0 < lambda_p_min < lambda_p_max and at least one step");
    CTL_CHECK(opts->amg_p_cycles >= 1 && opts->amg_p_nu >= 1 && opts->amg_p_max_levels >= 1, CTL_ERR_ARG,
              "ctl_stokes_pc_setup: bad AMG options");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    S->pc_ready = false;
    S->opts = *opts;
    CTL_TRY(ctl_pc_setup(h, &opts->velocity));
    // K_p hierarchy: K_p is singular (kernel = constants), the coarsest level gets a pseudo-inverse
    kp_free(S);
    auto from_hp = [&](int rc, const char *what) {       // errors of the pressure handle, reported on the velocity one
        if (rc != CTL_OK) ctl_set_error(h, std::string("ctl_stokes_pc_setup (") + what + "): " + hp->err);
        return rc;
    };
    AmgParams p;
    p.theta = opts->amg_p_theta;
    p.max_levels = opts->amg_p_max_levels;
    p.coarse_max = opts->amg_p_coarse_max;
    p.nu = opts->amg_p_nu;
    p.lo = opts->amg_p_lo;
    p.hi = opts->amg_p_hi;
    p.cycles = opts->amg_p_cycles;
    p.coarse = AMG_COARSE_PINV_CONSTANT;
    const int n_p = hp->n;
    {
        HostCSR Kp;
        Kp.n_rows = Kp.n_cols = n_p;
        Kp.indptr = hp->h_indptr;
        Kp.indices = hp->h_indices;
        Kp.values = S->h_Kp_solver.empty() ? hp->h_K[0] : S->h_Kp_solver;
        if (!S->fine_p) CTL_TRY(from_hp(sell_build_pattern(hp, hp->loc, S->fine_p), "SELL pattern"));
        if (h->cfg.world > 1) {                        // the exchange state the distributed hierarchy joins
            S->kp_x.reset(new PcState());
            CTL_TRY(from_hp(pc_mesh_exchange(hp, *S->kp_x), "K_p exchange geometry"));
        }
        S->Kp = AmgHierarchyDev();
        S->have_Kp = true;
        CTL_TRY(from_hp(amg_build(hp, Kp, p, S->fine_p, S->Kp, S->kp_x.get()), "K_p hierarchy"));
        if (S->kp_x) CTL_TRY(from_hp(halo_arena_finalize(hp, S->kp_x->arena), "K_p exchange arena"));
    }
    {
        const int rb = hp->row_begin, nl = hp->n_loc;
        std::vector<double> dinv(nl);
        for (int i = 0; i < nl; ++i) {
            const int r = rb + i;
            double d = 0.0;
            for (int k = hp->h_indptr[r]; k < hp->h_indptr[r + 1]; ++k)
                if (hp->h_indices[k] == r) d = hp->h_M[k];
            CTL_CHECK(d != 0.0, CTL_ERR_ARG, "ctl_stokes_pc_setup: pressure mass matrix has a zero diagonal entry");
            dinv[i] = 1.0 / d;
        }
        CTL_TRY(ctl_upload(h, &S->d_mp_dinv, dinv.data(), dinv.size()));
    }
    const size_t ts_bytes = 2ull * h->N * hp->n_loc * sizeof(double);
    if (!S->ts_b) CTL_CUDA(cudaMalloc((void **)&S->ts_b, ts_bytes));
    if (!S->ts_x) CTL_CUDA(cudaMalloc((void **)&S->ts_x, ts_bytes));
    CTL_CUDA(cudaMemsetAsync(S->ts_b, 0, ts_bytes, h->stream));
    CTL_CUDA(cudaMemsetAsync(S->ts_x, 0, ts_bytes, h->stream));
    CTL_CUDA(cudaStreamSynchronize(h->stream));
    S->pc_ready = true;
    return stokes_comm_check(S);
}

int ctl_stokes_apply(ctl_stokes S, const double *x, double *y)
{
    if (!S) return CTL_ERR_ARG;
    ctl_handle_s *h = S->hv;
    CTL_CHECK(x && y, CTL_ERR_ARG, "ctl_stokes_apply: null argument");
    CTL_TRY(with_tf(S, {x, nullptr}, y, [&](const double *xt, double *yt) { return stokes_apply_tf(S, xt, yt); }));
    return stokes_comm_check(S);
}

int ctl_stokes_pc_apply(ctl_stokes S, const double *b, double *u)
{
    if (!S) return CTL_ERR_ARG;
    ctl_handle_s *h = S->hv;
    CTL_CHECK(b && u, CTL_ERR_ARG, "ctl_stokes_pc_apply: null argument");
    CTL_TRY(with_tf(S, {b, nullptr}, u, [&](const double *bt, double *ut) { return stokes_pc_tf(S, bt, ut, true); }));
    return stokes_comm_check(S);
}

int ctl_stokes_pc_fn(ctl_stokes S, const double *b, double *u)
{
    if (!S) return CTL_ERR_ARG;
    ctl_handle_s *h = S->hv;
    CTL_CHECK(b && u, CTL_ERR_ARG, "ctl_stokes_pc_fn: null argument");
    CTL_TRY(with_tf(S, {b, nullptr}, u, [&](const double *bt, double *ut) { return stokes_pc_tf(S, bt, ut, false); }));
    return stokes_comm_check(S);
}

int ctl_stokes_set_pc_callback(ctl_stokes S, ctl_pc_callback fn, void *user)
{
    if (!S) return CTL_ERR_ARG;
    S->pc_cb = fn;
    S->pc_cb_user = user;
    return CTL_OK;
}

int ctl_stokes_solve(ctl_stokes S, const double *b, double *u, const ctl_krylov_options *opts, ctl_solve_result *result)
{
    if (!S) return CTL_ERR_ARG;
    ctl_handle_s *h = S->hv;
    CTL_CHECK(b && u && opts && result, CTL_ERR_ARG, "ctl_stokes_solve: null argument");
    CTL_CHECK(opts->ksp_type >= CTL_KSP_GMRES && opts->ksp_type <= CTL_KSP_MINRES, CTL_ERR_ARG,
              "ctl_stokes_solve: unknown ksp_type");
    CTL_CHECK(opts->pc >= CTL_PC_NONE && opts->pc <= CTL_PC_CALLBACK, CTL_ERR_ARG, "ctl_stokes_solve: unknown pc kind");
    if (opts->pc == CTL_PC_CALLBACK) CTL_CHECK(S->pc_cb, CTL_ERR_STATE, "ctl_stokes_solve: call ctl_stokes_set_pc_callback first");
    if (opts->pc == CTL_PC_BUILTIN) CTL_CHECK(S->pc_ready, CTL_ERR_STATE, "ctl_stokes_solve: call ctl_stokes_pc_setup first");
    CTL_TRY(with_tf(S, {b, u}, u, [&](const double *bt, double *ut) {
        StokesSolver K(S, *opts, *result);
        return krylov_solve(K, bt, ut);
    }));
    return stokes_comm_check(S);
}

int ctl_stokes_time(ctl_stokes S, int reps, double *out)
{
    if (!S) return CTL_ERR_ARG;
    ctl_handle_s *h = S->hv, *hp = S->hp;
    CTL_CHECK(out && reps > 0, CTL_ERR_ARG, "ctl_stokes_time: bad argument");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    Scratch xv, yv, xp;
    CTL_TRY(h->pool.take(&xv));
    CTL_TRY(h->pool.take(&yv));
    CTL_TRY(hp->pool.take(&xp));
    int rc = vec_zero(h, xv, h->vec_len());
    if (rc == CTL_OK) rc = vec_zero(h, yv, h->vec_len());
    if (rc == CTL_OK) rc = vec_zero(h, xp, hp->vec_len());
    EventPair ev;
    CTL_TRY(ev.create(h));
    const double tau = h->cfg.tau;
    float ms[2] = {0.f, 0.f};
    for (int which = 0; which < 2 && rc == CTL_OK; ++which) {
        for (int pass = 0; pass < 2 && rc == CTL_OK; ++pass) {        // pass 0 warms up
            cudaEventRecord(ev.begin, h->stream);
            for (int r = 0; r < reps && rc == CTL_OK; ++r) {        // several ranks: with the exchange of the ghosts
                rc = div_exchange(S, which == 1, which == 0 ? (const double *)xv : xp, 1);
                if (rc == CTL_OK)
                    rc = which == 0 ? panel_spmm(S, S->B, xv, S->d_ghost_v, nullptr, xp, tau, 1.0, T_TWO, T_NONE, false)
                                    : panel_spmm(S, S->BT, xp, S->d_ghost_p, nullptr, yv, tau, 1.0, T_ONE, T_NONE, true);
            }
            cudaEventRecord(ev.end, h->stream);
            cudaEventSynchronize(ev.end);
            cudaEventElapsedTime(&ms[which], ev.begin, ev.end);
        }
    }
    const double n_v = h->n_loc, n_p = hp->n_loc, N = h->N;
    std::vector<int> ptr_end(1);
    cudaMemcpy(ptr_end.data(), S->B.ptr + S->B.n_rows, sizeof(int), cudaMemcpyDeviceToHost);
    const double nnz = ptr_end[0];
    out[0] = ms[0] / reps;
    out[1] = 12.0 * nnz + 4.0 * (n_p + 1) + 8.0 * N * (n_v + n_p);
    out[2] = ms[1] / reps;
    out[3] = 12.0 * nnz + 4.0 * (n_v + 1) + 8.0 * N * (n_v + n_p) + 8.0 * N * n_v;
    CTL_TRY(rc);
    return stokes_comm_check(S);
}

}  // extern "C"
