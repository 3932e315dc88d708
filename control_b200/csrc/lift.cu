// Lifting of inhomogeneous, time-dependent Dirichlet data of the state into a right-hand side on the device
// (ctl_lift_bc, ctl_stokes_lift_bc).  The reference solves with homogenised conditions and moves the boundary
// values g_i into the right-hand sides through `v_inhom` (control/control.py:2993-3124 BE, 3137-3212 CN; the
// Stokes driver 3961-4243, divergence rows 4107-4128 / 4207-4228).  The lifting is affine in g and additive, so it
// runs as one separate pass over a homogeneous b (ctl_build_rhs, a host-built b, the b of ctl_nonlinear_residual):
//
//   b <- b - T(L(g)) on unconstrained rows (constrained rows untouched), with, per time block i,
//     BE  L_0[i] = tau M g_i (i < n_t - 1)          L_1[i] = tau K_i g_i + M g_i - M g_{i-1} (i > 0)
//     CN  L_0[i] = h M g_{i+1} + h M g_i (i >= 1)    L_1[i] = h K_{i+1} g_{i+1} + M g_{i+1} + h K_i g_i - M g_i (i >= 1)
//   h = tau / 2, T = (T_1, T_2) for CN and the identity for BE.
//
// Only entries of M / K in constrained COLUMNS contribute, so the data is a small boundary-column CSR: for each owned,
// unconstrained row with at least one constrained column, those entries of M and of K (one array, or n_t arrays when K
// is per level), and for each entry the position of its column in the ctl_set_bc list.  It is built on the host from
// the caller's full matrices on first use after ctl_assemble and dropped by ctl_set_values / ctl_set_bc /
// ctl_set_pattern, so the next call sees D_v at the current iterate.  One thread per such row walks all time blocks
// once, carries the previous level's products in registers and applies T in the same pass: the cost is
// O(rows next to the boundary x N), with no full-vector pass and no scratch vector.  Rows are local and every rank
// holds all n_t x n_bc values of g, so several ranks need no exchange.
#include <algorithm>

#include "common.cuh"

struct LiftState {
    int n_rows = 0;
    int levels = 1;                 // value sets of the second matrix (K): 1 or n_t; 0 = none (divergence rows)
    int64_t nnz = 0;
    int *d_rows = nullptr;          // local row of each boundary-adjacent row
    int *d_ptr = nullptr;           // [n_rows + 1]
    int *d_slot = nullptr;          // [nnz] column position in the ctl_set_bc list
    double *d_A = nullptr;          // [nnz] M (or B)
    double *d_K = nullptr;          // [levels][nnz] K
    ~LiftState()
    {
        cudaFree(d_rows);
        cudaFree(d_ptr);
        cudaFree(d_slot);
        cudaFree(d_A);
        cudaFree(d_K);
    }
};

namespace {

constexpr int LT = 128;

// (A g_l)[row], (K_l g_l)[row] over the constrained columns of one boundary-adjacent row
struct RowProducts {
    const int *slot;
    const double *A, *K;
    const double *g;
    int64_t k_stride;               // nnz (per-level K) or 0
    int n_bc, kb, ke;
    __device__ __forceinline__ void at(int l, double &ag, double &kg) const
    {
        ag = 0.0;
        kg = 0.0;
        const double *gl = g + (size_t)l * n_bc;
        const double *Kl = K + (size_t)l * k_stride;
        for (int e = kb; e < ke; ++e) {
            const double v = gl[__ldg(slot + e)];
            ag = fma(__ldg(A + e), v, ag);
            kg = fma(__ldg(Kl + e), v, kg);
        }
    }
};

// b_0[i] at b[base0 + i * step], b_1[i] at b[base1 + i * step]: block-major (step = n_loc) or time-fastest (step = 1)
template <bool CN>
__global__ void __launch_bounds__(LT) lift_kernel(const int *__restrict__ rows, const int *__restrict__ ptr,
                                                  const int *__restrict__ slot, const double *__restrict__ Mv,
                                                  const double *__restrict__ Kv, int64_t k_stride, const double *g,
                                                  int n_bc, double *b, int n_rows, int n_loc, int N, int tf, int ld,
                                                  double tau)
{
    const int t = blockIdx.x * LT + threadIdx.x;
    if (t >= n_rows) return;
    const int r = __ldg(rows + t);
    const RowProducts P{slot, Mv, Kv, g, k_stride, n_bc, __ldg(ptr + t), __ldg(ptr + t + 1)};
    const size_t step = tf ? 1 : (size_t)n_loc;
    double *b0 = b + (tf ? (size_t)r * ld : (size_t)r);
    double *b1 = b0 + (tf ? (size_t)n_loc * ld : (size_t)N * n_loc);
    double mg, kg;
    if (!CN) {                                          // N = n_t
        double mp = 0.0;                                // M g_{i-1}
        for (int i = 0; i < N; ++i) {
            P.at(i, mg, kg);
            if (i < N - 1) b0[i * step] -= tau * mg;
            b1[i * step] -= fma(tau, kg, mg) - mp;
            mp = mg;
        }
    } else {                                            // N = n_t - 1; D = -L before T
        const double hh = 0.5 * tau;
        double mp = 0.0, kp = 0.0, d0p = 0.0, d1p = 0.0;   // M g_i, K_i g_i, D_0[i-1], D_1[i-1]
        for (int i = 0; i < N; ++i) {
            P.at(i + 1, mg, kg);
            const double d0 = -hh * (mg + mp);
            const double d1 = -(fma(hh, kg, mg) + fma(hh, kp, -mp));
            b1[i * step] += d1 + d1p;                   // T_2: D_1[i] + D_1[i-1]
            if (i > 0) b0[(i - 1) * step] += d0p + d0;  // T_1: D_0[i-1] + D_0[i]
            d0p = d0;
            d1p = d1;
            mp = mg;
            kp = kg;
        }
        b0[(N - 1) * step] += d0p;
    }
}

// divergence rows of the outer Stokes vector (block-major, N blocks of n_p): D[i] = -tau (B g_{i (+1 for CN)})[row],
// b_1_0[i] += D[i] (+ D[i-1] for CN: T_2)
__global__ void __launch_bounds__(LT) lift_div_kernel(const int *__restrict__ rows, const int *__restrict__ ptr,
                                                      const int *__restrict__ slot, const double *__restrict__ Bv,
                                                      const double *g, int n_bc, double *b10, int n_rows, int n_p,
                                                      int N, int cn, double tau)
{
    const int t = blockIdx.x * LT + threadIdx.x;
    if (t >= n_rows) return;
    const int r = __ldg(rows + t), kb = __ldg(ptr + t), ke = __ldg(ptr + t + 1);
    double dp = 0.0;
    for (int i = 0; i < N; ++i) {
        const double *gl = g + (size_t)(cn ? i + 1 : i) * n_bc;
        double s = 0.0;
        for (int e = kb; e < ke; ++e) s = fma(__ldg(Bv + e), gl[__ldg(slot + e)], s);
        const double d = -tau * s;
        b10[(size_t)i * n_p + r] += cn ? d + dp : d;
        dp = d;
    }
}

// slot[c] = position of global column c in the ctl_set_bc list, -1 if unconstrained (a repeated dof keeps its last
// position, as numpy's `lift[:, bc_dofs] = g` does)
std::vector<int> bc_slots(const ctl_handle_s *h)
{
    std::vector<int> slot(h->n, -1);
    for (size_t i = 0; i < h->h_bc.size(); ++i) slot[h->h_bc[i]] = (int)i;
    return slot;
}

int upload_state(ctl_handle_s *h, LiftState &S, const std::vector<int> &rows, const std::vector<int> &ptr,
                 const std::vector<int> &slot, const std::vector<double> &A, const std::vector<double> &K)
{
    S.n_rows = (int)rows.size();
    S.nnz = (int64_t)slot.size();
    CTL_TRY(ctl_upload(h, &S.d_rows, rows.data(), rows.size()));
    CTL_TRY(ctl_upload(h, &S.d_ptr, ptr.data(), ptr.size()));
    CTL_TRY(ctl_upload(h, &S.d_slot, slot.data(), slot.size()));
    CTL_TRY(ctl_upload(h, &S.d_A, A.data(), A.size()));
    CTL_TRY(ctl_upload(h, &S.d_K, K.data(), K.size()));
    return CTL_OK;
}

// boundary-column CSR of this rank's rows from the host copies of M and K (the full values, before elimination)
int lift_build(ctl_handle_s *h)
{
    const std::vector<int> col_slot = bc_slots(h);
    const std::vector<int> &ip = h->h_indptr, &ix = h->h_indices;
    std::vector<int> rows, ptr(1, 0), slot;
    std::vector<int64_t> entry;                         // global CSR entry of each kept entry
    for (int r = 0; r < h->n_loc; ++r) {
        const int gr = h->row_begin + r;
        if (h->h_bcmask[gr]) continue;                  // constrained rows are left untouched
        for (int k = ip[gr]; k < ip[gr + 1]; ++k)
            if (col_slot[ix[k]] >= 0) {
                slot.push_back(col_slot[ix[k]]);
                entry.push_back(k);
            }
        if ((int)slot.size() > ptr.back()) {
            rows.push_back(r);
            ptr.push_back((int)slot.size());
        }
    }
    const size_t nnz = entry.size();
    const int levels = (int)h->h_K.size();
    std::vector<double> A(nnz), K(nnz * levels);
    for (size_t e = 0; e < nnz; ++e) {
        A[e] = h->h_M[entry[e]];
        for (int l = 0; l < levels; ++l) K[(size_t)l * nnz + e] = h->h_K[l][entry[e]];
    }
    auto S = std::make_shared<LiftState>();
    S->levels = levels;
    CTL_TRY(upload_state(h, *S, rows, ptr, slot, A, K));
    h->lift = S;
    return CTL_OK;
}

}  // namespace

void ctl_lift_invalidate(ctl_handle_s *h) { h->lift.reset(); }

int ctl_lift_div_setup(ctl_handle_s *h, const int32_t *B_indptr, const int32_t *B_indices, const double *B_values,
                       int row_begin, int n_rows, std::shared_ptr<LiftState> *out)
{
    const std::vector<int> col_slot = bc_slots(h);
    std::vector<int> rows, ptr(1, 0), slot;
    std::vector<double> A;
    for (int r = 0; r < n_rows; ++r) {
        for (int k = B_indptr[row_begin + r]; k < B_indptr[row_begin + r + 1]; ++k)
            if (col_slot[B_indices[k]] >= 0) {
                slot.push_back(col_slot[B_indices[k]]);
                A.push_back(B_values[k]);
            }
        if ((int)slot.size() > ptr.back()) {
            rows.push_back(r);
            ptr.push_back((int)slot.size());
        }
    }
    auto S = std::make_shared<LiftState>();
    S->levels = 0;
    CTL_TRY(upload_state(h, *S, rows, ptr, slot, A, std::vector<double>()));
    *out = S;
    return CTL_OK;
}

int ctl_lift_div_apply(ctl_handle_s *h, const LiftState *S, const double *g, double *b10, int n_p)
{
    if (!S || S->n_rows == 0 || h->h_bc.empty()) return CTL_OK;
    lift_div_kernel<<<ceil_div(S->n_rows, LT), LT, 0, h->stream>>>(S->d_rows, S->d_ptr, S->d_slot, S->d_A, g,
                                                                  (int)h->h_bc.size(), b10, S->n_rows, n_p, h->N,
                                                                  h->cfg.CN ? 1 : 0, h->cfg.tau);
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

extern "C" int ctl_lift_bc(ctl_handle h, const double *g, double *b, int layout)
{
    CTL_CHECK(h, CTL_ERR_ARG, "ctl_lift_bc: null handle");
    CTL_CHECK(layout == CTL_LAYOUT_BLOCK_MAJOR || layout == CTL_LAYOUT_TIME_FASTEST, CTL_ERR_ARG,
              "ctl_lift_bc: unknown layout");
    CTL_CHECK(h->assembled, CTL_ERR_STATE, "ctl_lift_bc: ctl_assemble has not been called");
    if (h->h_bc.empty()) return CTL_OK;
    CTL_CHECK(g && b, CTL_ERR_ARG, "ctl_lift_bc: null g or b (the handle has Dirichlet dofs)");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    if (!h->lift) CTL_TRY(lift_build(h));
    const LiftState &S = *h->lift;
    if (S.n_rows == 0) return CTL_OK;
    const int64_t k_stride = S.levels > 1 ? S.nnz : 0;
    const int tf = layout == CTL_LAYOUT_TIME_FASTEST ? 1 : 0;
    const int grid = ceil_div(S.n_rows, LT);
    const int n_bc = (int)h->h_bc.size();
    if (h->cfg.CN)
        lift_kernel<true><<<grid, LT, 0, h->stream>>>(S.d_rows, S.d_ptr, S.d_slot, S.d_A, S.d_K, k_stride, g, n_bc, b,
                                                      S.n_rows, h->n_loc, h->N, tf, h->ld, h->cfg.tau);
    else
        lift_kernel<false><<<grid, LT, 0, h->stream>>>(S.d_rows, S.d_ptr, S.d_slot, S.d_A, S.d_K, k_stride, g, n_bc, b,
                                                       S.n_rows, h->n_loc, h->N, tf, h->ld, h->cfg.tau);
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}
