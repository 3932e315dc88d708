// Discrete objective J_h on the device (SURVEY.md section 8c, "next" row f3):
//   J_h = 1/2 sum_i w_i (v_i - vhat_i)^T M (v_i - vhat_i) + 1/(2 beta) sum_i w_i zeta_i^T M zeta_i
// over the n_t time levels, trapezoid weights for CN, tau for BE (the row weights of block_00 /
// block_11, control/control.py:2915-2923, 2940-2953; the reference itself never evaluates J).
// One kernel over (rows x levels) with the FULL mass matrix (no Dirichlet elimination: vhat need not
// vanish on the boundary), fixed-order two-stage reduction, 2 n_t doubles read back.
//
// Several ranks (round 2): every rank hands over ITS rows of the level-major arrays (n_t x n_local).  The products
// with M gather ghost columns, so the arrays are first extended to n_t x (n_local + n_halo) -- owned entries copied,
// ghost entries fetched from their owners with the row exchange of the batched kernels (levels travel as the
// columns of a time-fastest panel, comm.cu) -- and the same kernels run on the local pattern, whose column
// numbering is exactly that (owned columns first, ghosts behind).  Scalars are all-reduced.
#include "common.cuh"

namespace {

constexpr int QT = 256;

__global__ void __launch_bounds__(QT) quadform_partial_kernel(const int *__restrict__ ptr, const int *__restrict__ cols,
                                                             const double *__restrict__ Mv, const double *__restrict__ v,
                                                             const double *__restrict__ zeta,
                                                             const double *__restrict__ vhat, double *__restrict__ partial,
                                                             int n, int stride)
{
    __shared__ double sh[2][QT / 32];
    const size_t base = (size_t)blockIdx.y * stride;      // n rows of this rank; stride = n + ghost entries
    const int row = blockIdx.x * QT + threadIdx.x;
    double qd = 0.0, qz = 0.0;
    if (row < n) {
        double ad = 0.0, az = 0.0;
        for (int k = ptr[row]; k < ptr[row + 1]; ++k) {
            const int c = cols[k];
            const double m = Mv[k];
            ad = fma(m, v[base + c] - vhat[base + c], ad);
            az = fma(m, zeta[base + c], az);
        }
        qd = (v[base + row] - vhat[base + row]) * ad;
        qz = zeta[base + row] * az;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        qd += __shfl_xor_sync(0xffffffffu, qd, o);
        qz += __shfl_xor_sync(0xffffffffu, qz, o);
    }
    if ((threadIdx.x & 31) == 0) {
        sh[0][threadIdx.x >> 5] = qd;
        sh[1][threadIdx.x >> 5] = qz;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
        for (int w = 0; w < QT / 32; ++w) {
            a += sh[0][w];
            b += sh[1][w];
        }
        double *p = partial + 2 * ((size_t)blockIdx.y * gridDim.x + blockIdx.x);
        p[0] = a;
        p[1] = b;
    }
}

// out[level][0..1] = sums over the row blocks, in block order
__global__ void quadform_finish_kernel(const double *__restrict__ partial, double *__restrict__ out, int blocks)
{
    if (threadIdx.x >= 2) return;
    const double *p = partial + 2 * (size_t)blockIdx.x * blocks + threadIdx.x;
    double s = 0.0;
    for (int b = 0; b < blocks; ++b) s += p[2 * (size_t)b];
    out[2 * blockIdx.x + threadIdx.x] = s;
}

// panel[r][j] = x[(l0 + j) * n + r] for j < cnt, 0 otherwise (levels of a level-major array as panel columns)
__global__ void levels_to_panel_kernel(const double *__restrict__ x, int l0, int cnt, int n, int ld, double *__restrict__ panel)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)n * ld) return;
    const int r = (int)(idx / ld), j = (int)(idx % ld);
    panel[idx] = j < cnt ? x[(size_t)(l0 + j) * n + r] : 0.0;
}

// ext[(l0 + j) * stride + n + g] = halo[g][j]: ghost entries behind the owned ones
__global__ void halo_to_levels_kernel(const double *__restrict__ halo, int l0, int cnt, int n_halo, int ld, int n, int stride,
                                      double *__restrict__ ext)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)n_halo * cnt) return;
    const int g = (int)(idx / cnt), j = (int)(idx % cnt);
    ext[(size_t)(l0 + j) * stride + n + g] = halo[(size_t)g * ld + j];
}

}  // namespace

// L levels of this rank's rows -> L levels of (n_loc + n_halo) entries in local column numbering (ext: device,
// allocated by the caller).  One rank: ext is not needed (callers pass the array itself with stride n).
static int extend_levels(ctl_handle_s *h, const double *x_loc, int L, double *ext)
{
    const int nl = h->n_loc, nh = h->n_halo, ld = h->ld, stride = nl + nh;
    CTL_CUDA(cudaMemcpy2DAsync(ext, (size_t)stride * sizeof(double), x_loc, (size_t)nl * sizeof(double),
                               (size_t)nl * sizeof(double), (size_t)L, cudaMemcpyDeviceToDevice, h->stream));
    if (nh == 0) return CTL_OK;
    Scratch panel;
    CTL_TRY(h->pool.take(&panel));
    for (int l0 = 0; l0 < L; l0 += ld) {
        const int cnt = std::min(ld, L - l0);
        levels_to_panel_kernel<<<ceil_div((int64_t)nl * ld, 256), 256, 0, h->stream>>>(x_loc, l0, cnt, nl, ld, panel);
        h->launches++;
        CTL_TRY(ctl_halo_exchange_panel(h, panel));
        halo_to_levels_kernel<<<ceil_div((int64_t)nh * cnt, 256), 256, 0, h->stream>>>(h->d_halo, l0, cnt, nh, ld, nl, stride, ext);
        h->launches++;
        if (cudaGetLastError() != cudaSuccess) {
            ctl_set_error(h, "extend_levels: CUDA failure");
            return CTL_ERR_CUDA;
        }
    }
    return CTL_OK;
}

extern "C" int ctl_objective(ctl_handle h, const double *v, const double *zeta, const double *v_hat, double *out)
{
    CTL_CHECK(h && v && zeta && v_hat && out, CTL_ERR_ARG, "ctl_objective: null argument");
    CTL_CHECK(h->assembled, CTL_ERR_STATE, "ctl_objective: ctl_assemble has not been called");
    CTL_CHECK(h->cfg.world == 1 || h->comm, CTL_ERR_STATE, "ctl_objective: call ctl_comm_init first (world > 1)");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    const int n = h->n_loc, n_t = h->cfg.n_t, stride = h->n_loc + h->n_halo;
    if (!h->d_M_full) {
        std::vector<double> buf(h->loc_entry.size());
        for (size_t p = 0; p < buf.size(); ++p) buf[p] = h->h_M[h->loc_entry[p]];
        CTL_TRY(ctl_upload(h, &h->d_M_full, buf.data(), buf.size()));
    }
    const int blocks = ceil_div(n, QT);
    DeviceArray<double> partial, sums, ext;
    int rc = CTL_OK;
    cudaError_t e = cudaSuccess;
    std::vector<double> hs(2 * (size_t)n_t);
    do {
        const double *pv = v, *pz = zeta, *ph = v_hat;
        if (h->n_halo > 0) {      // several ranks: ghost entries of the three arrays behind the owned ones
            const size_t one = (size_t)n_t * stride;
            if ((e = ext.alloc(3 * one)) != cudaSuccess) break;
            if ((rc = extend_levels(h, v, n_t, ext)) != CTL_OK) break;
            if ((rc = extend_levels(h, zeta, n_t, ext + one)) != CTL_OK) break;
            if ((rc = extend_levels(h, v_hat, n_t, ext + 2 * one)) != CTL_OK) break;
            pv = ext;
            pz = ext + one;
            ph = ext + 2 * one;
        }
        if ((e = partial.alloc(2 * (size_t)blocks * n_t)) != cudaSuccess) break;
        if ((e = sums.alloc(2 * n_t)) != cudaSuccess) break;
        quadform_partial_kernel<<<dim3(blocks, n_t), QT, 0, h->stream>>>(h->d_indptr, h->d_indices, h->d_M_full, pv, pz, ph,
                                                                        partial, n, h->n_halo > 0 ? stride : n);
        quadform_finish_kernel<<<n_t, 32, 0, h->stream>>>(partial, sums, blocks);
        h->launches += 2;
        if ((rc = ctl_allreduce_sum(h, sums, 2 * n_t)) != CTL_OK) break;      // (no-op on one rank)
        e = cudaMemcpyAsync(hs.data(), sums, sizeof(double) * hs.size(), cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    } while (0);
    if (e != cudaSuccess) {
        ctl_set_error(h, std::string("ctl_objective: ") + cudaGetErrorString(e));
        return CTL_ERR_CUDA;
    }
    if (rc != CTL_OK) return rc;
    const double tau = h->cfg.tau, beta = h->cfg.beta;
    double J = 0.0;
    for (int i = 0; i < n_t; ++i) {
        const double w = (h->cfg.CN && (i == 0 || i == n_t - 1)) ? 0.5 * tau : tau;
        J += 0.5 * w * hs[2 * i];
        J += 0.5 / beta * w * hs[2 * i + 1];
    }
    *out = J;
    return CTL_OK;
}

// ---------------------------------------------------------------------------------------------
// Right-hand sides of linear_solve from NODAL data on the device (SURVEY.md "next" row f3;
// control/control.py:2980-3243 for homogeneous Dirichlet data).  In the reference v_d and f are
// cofunctions assembled by Firedrake, one FE assembly per time level; for data interpolated into the
// space (README.md:33-60 and every test) they equal M v_hat_i and M f_i, so only nodal values need to
// cross the boundary.  Block-major = level-major here, so every step is one kernel over rows x blocks.
// ---------------------------------------------------------------------------------------------
namespace {

// out[i][r] = alpha * sum_k M[r,k] (x[i + off][k] + (pair ? x[i + off + 1][k] : 0)); constrained rows 0
__global__ void __launch_bounds__(QT) rhs_rows_kernel(const int *__restrict__ ptr, const int *__restrict__ cols,
                                                     const double *__restrict__ Mv, const uint8_t *__restrict__ bc,
                                                     const double *__restrict__ x, double *__restrict__ out, int n,
                                                     int stride, double alpha, int pair, int off)
{
    const int row = blockIdx.x * QT + threadIdx.x;
    if (row >= n) return;
    const int i = blockIdx.y;
    double acc = 0.0;
    if (!bc[row]) {
        const double *x0 = x + (size_t)(i + off) * stride, *x1 = x0 + stride;      // stride = n + ghost entries
        for (int k = ptr[row]; k < ptr[row + 1]; ++k) {
            const int c = cols[k];
            acc = fma(Mv[k], pair ? x0[c] + x1[c] : x0[c], acc);
        }
        acc *= alpha;
    }
    out[(size_t)i * n + row] = acc;
}

// out[i] = in[i] + in[i + 1] (mode 1: T_1) / in[i] + in[i - 1] (mode 2: T_2) over N blocks of n
__global__ void bm_time_transform_kernel(const double *__restrict__ in, double *__restrict__ out, int n, int N, int mode)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)N * n) return;
    const int i = (int)(idx / n);
    double v = in[idx];
    if (mode == 1 && i + 1 < N) v += in[idx + n];
    if (mode == 2 && i > 0) v += in[idx - n];
    out[idx] = v;
}

// y[r] -= c[r] on unconstrained rows of one block
__global__ void block_sub_kernel(double *__restrict__ y, const double *__restrict__ c, const uint8_t *__restrict__ bc, int n)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n && !bc[r]) y[r] -= c[r];
}

}  // namespace

extern "C" int ctl_build_rhs(ctl_handle h, const double *v_hat, const double *f_nodal, const double *v_0_host, double *b)
{
    CTL_CHECK(h && v_hat && f_nodal && b, CTL_ERR_ARG, "ctl_build_rhs: null argument");
    CTL_CHECK(h->assembled, CTL_ERR_STATE, "ctl_build_rhs: ctl_assemble has not been called");
    CTL_CHECK(h->cfg.world == 1 || h->comm, CTL_ERR_STATE, "ctl_build_rhs: call ctl_comm_init first (world > 1)");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    const int n = h->n_loc, n_t = h->cfg.n_t, N = h->N, rb = h->row_begin;
    const int stride = h->n_halo > 0 ? h->n_loc + h->n_halo : n;
    const bool cn = h->cfg.CN != 0;
    const double tau = h->cfg.tau;
    if (!h->d_M_full) {
        std::vector<double> buf(h->loc_entry.size());
        for (size_t p = 0; p < buf.size(); ++p) buf[p] = h->h_M[h->loc_entry[p]];
        CTL_TRY(ctl_upload(h, &h->d_M_full, buf.data(), buf.size()));
    }
    DeviceArray<double> ext;
    const double *pv = v_hat, *pf = f_nodal;
    if (h->n_halo > 0) {      // several ranks: this rank's rows of the nodal data + the ghost entries the products gather
        const size_t one = (size_t)n_t * stride;
        CTL_CUDA(ext.alloc(2 * one));
        CTL_TRY(extend_levels(h, v_hat, n_t, ext));
        CTL_TRY(extend_levels(h, f_nodal, n_t, ext + one));
        pv = ext;
        pf = ext + one;
    }
    const int blocks = ceil_div(n, QT);
    const size_t half = (size_t)N * n;
    Scratch work;                           // untransformed rows (CN) before T_1 / T_2
    CTL_TRY(h->pool.take(&work));           // a scratch vector holds at least 2 N n doubles
    double *r0 = cn ? work : b, *r1 = cn ? work + half : b + half;
    // M-weighted rows: CN h M (x_i + x_{i+1}), i < N;  BE tau M x_i, with b_0 row n_t - 1 = 0 and b_1 row 0 from v_0
    const double alpha = cn ? 0.5 * tau : tau;
    rhs_rows_kernel<<<dim3(blocks, N), QT, 0, h->stream>>>(h->d_indptr, h->d_indices, h->d_M_full, h->d_bcmask, pv, r0, n,
                                                          stride, alpha, cn ? 1 : 0, 0);
    rhs_rows_kernel<<<dim3(blocks, N), QT, 0, h->stream>>>(h->d_indptr, h->d_indices, h->d_M_full, h->d_bcmask, pf, r1, n,
                                                          stride, alpha, cn ? 1 : 0, 0);
    h->launches += 2;
    int rc = CTL_OK;
    if (!cn) {
        if (cudaMemsetAsync(r0 + (size_t)(n_t - 1) * n, 0, (size_t)n * sizeof(double), h->stream) != cudaSuccess ||
            cudaMemsetAsync(r1, 0, (size_t)n * sizeof(double), h->stream) != cudaSuccess)
            rc = CTL_ERR_CUDA;
    }
    // terms of the initial condition (control/control.py:3000-3004 BE, 3217-3240 CN), on the host:
    // two products with one n-vector (v_0: all n entries on every rank; the rows of this rank are computed)
    if (rc == CTL_OK && v_0_host) {
        const std::vector<double> &K0 = h->h_K[0];
        std::vector<double> c0(n, 0.0), c1(n, 0.0);
        for (int r = 0; r < n; ++r) {
            const int g = rb + r;
            double mv = 0.0, kv = 0.0;
            for (int k = h->h_indptr[g]; k < h->h_indptr[g + 1]; ++k) {
                const double x = v_0_host[h->h_indices[k]];
                mv += h->h_M[k] * x;
                kv += K0[k] * x;
            }
            if (cn) {
                c0[r] = 0.5 * tau * mv;                 // b_0[0] -= h M v_0
                c1[r] = 0.5 * tau * kv - mv;            // b_1[0] -= (h K_0 - M) v_0
            } else {
                c1[r] = -(tau * kv + mv);               // b_1[0]  = (tau K_0 + M) v_0
            }
        }
        DeviceArray<double> d_c;
        if (d_c.alloc(2 * (size_t)n) != cudaSuccess) rc = CTL_ERR_CUDA;
        if (rc == CTL_OK) {
            cudaMemcpyAsync(d_c, c0.data(), (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream);
            cudaMemcpyAsync(d_c + n, c1.data(), (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream);
            if (cn) block_sub_kernel<<<ceil_div(n, 256), 256, 0, h->stream>>>(r0, d_c, h->d_bcmask, n);
            block_sub_kernel<<<ceil_div(n, 256), 256, 0, h->stream>>>(r1, d_c + n, h->d_bcmask, n);
            h->launches += cn ? 2 : 1;
            cudaStreamSynchronize(h->stream);           // c0 / c1 are host temporaries
        }
    }
    if (rc == CTL_OK && cn) {                           // b_0 = T_1 rows, b_1 = T_2 rows (3242-3243)
        const int tb = ceil_div((int64_t)half, 256);
        bm_time_transform_kernel<<<tb, 256, 0, h->stream>>>(r0, b, n, N, 1);
        bm_time_transform_kernel<<<tb, 256, 0, h->stream>>>(r1, b + half, n, N, 2);
        h->launches += 2;
    }
    if (rc == CTL_OK && cudaGetLastError() != cudaSuccess) rc = CTL_ERR_CUDA;
    if (rc == CTL_OK && ext && cudaStreamSynchronize(h->stream) != cudaSuccess) rc = CTL_ERR_CUDA;      // ext is freed on return
    if (rc != CTL_OK) ctl_set_error(h, "ctl_build_rhs: CUDA failure");
    return rc;
}
