// Krylov vector work (SURVEY.md row K5): what PETSc does through VecMDot / VecMAXPY /
// VecNorm / VecAXPY inside KSPSolve (preconditioner/preconditioner.py:758-759).
//
// Every kernel is a single streaming pass with 16-byte loads, warp-shuffle reductions and
// a deterministic two-stage (per-block partials, then one block) final reduction, so a
// solve is reproducible run to run.  Scalars that only feed the next kernel (Gram-Schmidt
// coefficients, the new basis vector's norm) stay in device memory: one host
// synchronisation per Krylov iteration.  On several GPUs the partial results are
// all-reduced on the stream (comm.cu) before anyone reads them.
#include <algorithm>
#include <cstring>

#include "common.cuh"
#include "vec_ops.cuh"

namespace {

constexpr int RB = 1024;            // reduction grid (blocks), >= 148 * resident CTAs
constexpr int RT = 256;             // threads per block
constexpr int MAXK = 256;           // most vectors in one multi-dot / maxpy (GMRES restart + 2)

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// block-wide sums of KC values; result valid in thread 0
template <int KC>
__device__ __forceinline__ void block_sum(double (&acc)[KC], double *smem /* KC * 8 */)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < KC; ++j) {
        acc[j] = warp_sum(acc[j]);
        if (lane == 0) smem[j * (RT / 32) + w] = acc[j];
    }
    __syncthreads();
    if (w == 0) {
#pragma unroll
        for (int j = 0; j < KC; ++j) {
            double v = lane < RT / 32 ? smem[j * (RT / 32) + lane] : 0.0;
            acc[j] = warp_sum(v);
        }
    }
}

struct Ptrs8 {
    const double *p[8];
};

// partial[j * gridDim.x + block] = sum over this block's elements of V_j * w
__global__ void __launch_bounds__(RT) multi_dot_kernel(Ptrs8 V, int kc, const double *__restrict__ w,
                                                      int64_t len2, double *__restrict__ partial)
{
    __shared__ double smem[8 * (RT / 32)];
    double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const double2 *w2 = reinterpret_cast<const double2 *>(w);
    for (int64_t i = (int64_t)blockIdx.x * RT + threadIdx.x; i < len2; i += (int64_t)gridDim.x * RT) {
        const double2 wi = w2[i];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (j < kc) {
                const double2 v = reinterpret_cast<const double2 *>(V.p[j])[i];
                acc[j] = fma(v.x, wi.x, fma(v.y, wi.y, acc[j]));
            }
        }
    }
    block_sum<8>(acc, smem);
    if (threadIdx.x == 0)
        for (int j = 0; j < kc; ++j) partial[(size_t)j * gridDim.x + blockIdx.x] = acc[j];
}

// out[j] = sum_b partial[j * nb + b]; optionally out_sqrt[j] = sqrt(out[j])
__global__ void __launch_bounds__(RT) final_sum_kernel(const double *__restrict__ partial, int nb,
                                                      double *__restrict__ out, double *__restrict__ out_sqrt)
{
    __shared__ double smem[RT / 32];
    const int j = blockIdx.x;
    double acc[1] = {0.0};
    for (int b = threadIdx.x; b < nb; b += RT) acc[0] += partial[(size_t)j * nb + b];
    block_sum<1>(acc, smem);
    if (threadIdx.x == 0) {
        out[j] = acc[0];
        if (out_sqrt) out_sqrt[j] = sqrt(acc[0]);
    }
}

// w += sign * sum_j coef[j] V_j ; partial[block] = sum of w_new^2 over the block
__global__ void __launch_bounds__(RT) maxpy_kernel(double *__restrict__ w, Ptrs8 V, int kc,
                                                  const double *__restrict__ coef, double sign,
                                                  int64_t len2, double *__restrict__ partial)
{
    __shared__ double smem[RT / 32];
    double c[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) c[j] = j < kc ? sign * coef[j] : 0.0;
    double acc[1] = {0.0};
    double2 *w2 = reinterpret_cast<double2 *>(w);
    for (int64_t i = (int64_t)blockIdx.x * RT + threadIdx.x; i < len2; i += (int64_t)gridDim.x * RT) {
        double2 wi = w2[i];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (j < kc) {
                const double2 v = reinterpret_cast<const double2 *>(V.p[j])[i];
                wi.x = fma(c[j], v.x, wi.x);
                wi.y = fma(c[j], v.y, wi.y);
            }
        }
        w2[i] = wi;
        acc[0] = fma(wi.x, wi.x, fma(wi.y, wi.y, acc[0]));
    }
    if (partial) {
        block_sum<1>(acc, smem);
        if (threadIdx.x == 0) partial[blockIdx.x] = acc[0];
    }
}

// dst = a * x + b * y (+ c * z); a, b, c scaled by 1 / *inv_scalar when given
// (operands may alias dst element-wise: no __restrict__)
__global__ void __launch_bounds__(RT) lincomb_kernel(double *dst, double a, const double *x, double b,
                                                    const double *y, double c, const double *z,
                                                    const double *inv_scalar, int64_t len2)
{
    if (inv_scalar) {
        const double s = 1.0 / *inv_scalar;
        a *= s;
        b *= s;
        c *= s;
    }
    double2 *d2 = reinterpret_cast<double2 *>(dst);
    for (int64_t i = (int64_t)blockIdx.x * RT + threadIdx.x; i < len2; i += (int64_t)gridDim.x * RT) {
        double2 r = make_double2(0.0, 0.0);
        if (x) {
            const double2 v = reinterpret_cast<const double2 *>(x)[i];
            r.x = a * v.x;
            r.y = a * v.y;
        }
        if (y) {
            const double2 v = reinterpret_cast<const double2 *>(y)[i];
            r.x = fma(b, v.x, r.x);
            r.y = fma(b, v.y, r.y);
        }
        if (z) {
            const double2 v = reinterpret_cast<const double2 *>(z)[i];
            r.x = fma(c, v.x, r.x);
            r.y = fma(c, v.y, r.y);
        }
        d2[i] = r;
    }
}

// y += c r, then partial[block] = sum over the block of v * y_new: the update of vec_lincomb(y, 1, y, c, r) (1 * y is
// exact) followed by multi_dot_kernel's loop for V = {v}, w = y; block_sum<1> adds what block_sum<8> adds for j = 0
__global__ void __launch_bounds__(RT) axpy_dot_kernel(double *y, double c, const double *r, const double *v,
                                                     int64_t len2, double *__restrict__ partial)
{
    __shared__ double smem[RT / 32];
    double acc[1] = {0.0};
    double2 *y2 = reinterpret_cast<double2 *>(y);
    for (int64_t i = (int64_t)blockIdx.x * RT + threadIdx.x; i < len2; i += (int64_t)gridDim.x * RT) {
        double2 yi = y2[i];
        const double2 ri = reinterpret_cast<const double2 *>(r)[i];
        yi.x = fma(c, ri.x, yi.x);
        yi.y = fma(c, ri.y, yi.y);
        y2[i] = yi;
        const double2 vi = reinterpret_cast<const double2 *>(v)[i];
        acc[0] = fma(vi.x, yi.x, fma(vi.y, yi.y, acc[0]));
    }
    block_sum<1>(acc, smem);
    if (threadIdx.x == 0) partial[blockIdx.x] = acc[0];
}

// MINRES direction, iterate and next Lanczos vector in one pass, each as its own vec_lincomb computes it:
// w_new = a v + b w2 + c w; x += phi w_new; then, when y is given, v = s y.  Every element of v is read before the
// same thread overwrites it.
__global__ void __launch_bounds__(RT) minres_update_kernel(double *w_new, double a, const double *v, double b,
                                                          const double *w2, double c, const double *w, double *x,
                                                          double phi, double *v_next, double s, const double *y,
                                                          int64_t len2)
{
    for (int64_t i = (int64_t)blockIdx.x * RT + threadIdx.x; i < len2; i += (int64_t)gridDim.x * RT) {
        const double2 vi = reinterpret_cast<const double2 *>(v)[i];
        const double2 w2i = reinterpret_cast<const double2 *>(w2)[i];
        const double2 wi = reinterpret_cast<const double2 *>(w)[i];
        double2 r;
        r.x = fma(c, wi.x, fma(b, w2i.x, a * vi.x));
        r.y = fma(c, wi.y, fma(b, w2i.y, a * vi.y));
        reinterpret_cast<double2 *>(w_new)[i] = r;
        double2 xi = reinterpret_cast<double2 *>(x)[i];
        xi.x = fma(phi, r.x, xi.x);
        xi.y = fma(phi, r.y, xi.y);
        reinterpret_cast<double2 *>(x)[i] = xi;
        if (y) {
            const double2 yi = reinterpret_cast<const double2 *>(y)[i];
            reinterpret_cast<double2 *>(v_next)[i] = make_double2(s * yi.x, s * yi.y);
        }
    }
}

// partial[block] = sum over the block of |x|
__global__ void __launch_bounds__(RT) asum_kernel(const double *x, int64_t len2, double *__restrict__ partial)
{
    __shared__ double smem[RT / 32];
    double acc[1] = {0.0};
    for (int64_t i = (int64_t)blockIdx.x * RT + threadIdx.x; i < len2; i += (int64_t)gridDim.x * RT) {
        const double2 xi = reinterpret_cast<const double2 *>(x)[i];
        acc[0] += fabs(xi.x) + fabs(xi.y);
    }
    block_sum<1>(acc, smem);
    if (threadIdx.x == 0) partial[blockIdx.x] = acc[0];
}

int grid_for(int64_t len2)
{
    int64_t b = (len2 + RT - 1) / RT;
    return (int)std::max<int64_t>(1, std::min<int64_t>(b, RB));
}

}  // namespace

int vec_workspace(ctl_handle_s *h, double **partials, double **scalars)
{
    // lives with the handle: MAXK * RB partials + 2 * MAXK scalar slots
    static_assert(RB >= 1, "");
    if (!h->d_red) {
        CTL_CUDA(cudaMalloc((void **)&h->d_red, (size_t)(MAXK * RB + 2 * MAXK) * sizeof(double)));
        CTL_CUDA(cudaMallocHost((void **)&h->h_red, 2 * MAXK * sizeof(double)));
    }
    *partials = h->d_red;
    *scalars = h->d_red + MAXK * RB;
    return CTL_OK;
}

int vec_zero(ctl_handle_s *h, double *x, int64_t len)
{
    CTL_CUDA(cudaMemsetAsync(x, 0, len * sizeof(double), h->stream));
    return CTL_OK;
}

int vec_copy(ctl_handle_s *h, double *dst, const double *src, int64_t len)
{
    if (dst != src)
        CTL_CUDA(cudaMemcpyAsync(dst, src, len * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    return CTL_OK;
}

int vec_lincomb(ctl_handle_s *h, double *dst, double a, const double *x, double b, const double *y,
                double c, const double *z, const double *inv_scalar_dev, int64_t len)
{
    const int64_t len2 = len / 2;
    lincomb_kernel<<<grid_for(len2), RT, 0, h->stream>>>(
        dst, a, x, b, y, c, z, inv_scalar_dev, len2);
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

int vec_multi_dot_dev(ctl_handle_s *h, const double *const *V, int k, const double *w, int64_t len,
                      double *out_dev, double *out_sqrt_dev)
{
    double *partials, *scalars;
    CTL_TRY(vec_workspace(h, &partials, &scalars));
    CTL_CHECK(k <= MAXK, CTL_ERR_ARG, "vec_multi_dot: too many vectors");
    const int64_t len2 = len / 2;
    const int nb = grid_for(len2);
    for (int j0 = 0; j0 < k; j0 += 8) {
        Ptrs8 P;
        const int kc = std::min(8, k - j0);
        for (int j = 0; j < 8; ++j) P.p[j] = j < kc ? V[j0 + j] : nullptr;
        multi_dot_kernel<<<nb, RT, 0, h->stream>>>(P, kc, w, len2, partials + (size_t)j0 * nb);
        h->launches++;
    }
    final_sum_kernel<<<k, RT, 0, h->stream>>>(partials, nb, out_dev, h->comm ? nullptr : out_sqrt_dev);
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    if (h->comm) {
        CTL_TRY(ctl_allreduce_sum(h, out_dev, k));
        if (out_sqrt_dev) CTL_TRY(vec_sqrt_dev(h, out_dev, out_sqrt_dev, k));
    }
    return CTL_OK;
}

namespace {
__global__ void sqrt_kernel(const double *in, double *out, int k)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < k) out[i] = sqrt(in[i]);
}
}  // namespace

int vec_sqrt_dev(ctl_handle_s *h, const double *in, double *out, int k)
{
    sqrt_kernel<<<1, 64, 0, h->stream>>>(in, out, k);
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

int vec_maxpy_dev(ctl_handle_s *h, double *w, const double *const *V, int k, const double *coef_dev,
                  double sign, int64_t len, double *norm2_dev, double *norm_dev)
{
    double *partials, *scalars;
    CTL_TRY(vec_workspace(h, &partials, &scalars));
    const int64_t len2 = len / 2;
    const int nb = grid_for(len2);
    for (int j0 = 0; j0 < k || (k == 0 && j0 == 0); j0 += 8) {
        Ptrs8 P;
        const int kc = std::max(0, std::min(8, k - j0));
        for (int j = 0; j < 8; ++j) P.p[j] = j < kc ? V[j0 + j] : nullptr;
        const bool lastpass = j0 + 8 >= k;
        maxpy_kernel<<<nb, RT, 0, h->stream>>>(w, P, kc, coef_dev + j0, sign, len2,
                                               (lastpass && norm2_dev) ? partials : nullptr);
        h->launches++;
    }
    if (norm2_dev) {
        final_sum_kernel<<<1, RT, 0, h->stream>>>(partials, nb, norm2_dev, h->comm ? nullptr : norm_dev);
        h->launches++;
        if (h->comm) {
            CTL_TRY(ctl_allreduce_sum(h, norm2_dev, 1));
            if (norm_dev) CTL_TRY(vec_sqrt_dev(h, norm2_dev, norm_dev, 1));
        }
    }
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

int vec_maxpy_host(ctl_handle_s *h, double *w, const double *const *V, int k, const double *coef_host,
                   double sign, int64_t len)
{
    double *partials, *scalars;
    CTL_TRY(vec_workspace(h, &partials, &scalars));
    CTL_CHECK(k <= MAXK, CTL_ERR_ARG, "vec_maxpy: too many vectors");
    // stage the coefficients in the second half of the scalar area
    CTL_CUDA(cudaStreamSynchronize(h->stream));
    memcpy(h->h_red + MAXK, coef_host, k * sizeof(double));
    CTL_CUDA(cudaMemcpyAsync(scalars + MAXK, h->h_red + MAXK, k * sizeof(double), cudaMemcpyHostToDevice,
                             h->stream));
    return vec_maxpy_dev(h, w, V, k, scalars + MAXK, sign, len, nullptr, nullptr);
}

int vec_read_scalars(ctl_handle_s *h, const double *dev, int k, double *host_out)
{
    CTL_CUDA(cudaMemcpyAsync(h->h_red, dev, k * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CTL_CUDA(cudaStreamSynchronize(h->stream));
    memcpy(host_out, h->h_red, k * sizeof(double));
    return CTL_OK;
}

int vec_dot_host(ctl_handle_s *h, const double *x, const double *y, int64_t len, double *out)
{
    double *partials, *scalars;
    CTL_TRY(vec_workspace(h, &partials, &scalars));
    const double *V[1] = {x};
    CTL_TRY(vec_multi_dot_dev(h, V, 1, y, len, scalars, nullptr));
    return vec_read_scalars(h, scalars, 1, out);
}

int vec_norm_host(ctl_handle_s *h, const double *x, int64_t len, double *out)
{
    double d = 0;
    CTL_TRY(vec_dot_host(h, x, x, len, &d));
    *out = sqrt(d);
    return CTL_OK;
}

// the block partials in partials[0, nb) -> their sum on the host, all-reduced over the ranks
static int sum_partials_host(ctl_handle_s *h, int nb, double *out)
{
    double *partials, *scalars;
    CTL_TRY(vec_workspace(h, &partials, &scalars));
    final_sum_kernel<<<1, RT, 0, h->stream>>>(partials, nb, scalars, nullptr);
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    if (h->comm) CTL_TRY(ctl_allreduce_sum(h, scalars, 1));
    return vec_read_scalars(h, scalars, 1, out);
}

int vec_axpy_dot_host(ctl_handle_s *h, double *y, double c, const double *r, const double *v, int64_t len,
                      double *out)
{
    double *partials, *scalars;
    CTL_TRY(vec_workspace(h, &partials, &scalars));
    const int64_t len2 = len / 2;
    axpy_dot_kernel<<<grid_for(len2), RT, 0, h->stream>>>(y, c, r, v, len2, partials);
    h->launches++;
    return sum_partials_host(h, grid_for(len2), out);
}

int vec_minres_update(ctl_handle_s *h, double *w_new, double a, const double *v, double b, const double *w2,
                      double c, const double *w, double *x, double phi, double *v_next, double s, const double *y,
                      int64_t len)
{
    const int64_t len2 = len / 2;
    minres_update_kernel<<<grid_for(len2), RT, 0, h->stream>>>(w_new, a, v, b, w2, c, w, x, phi, v_next, s, y, len2);
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

int vec_is_zero_host(ctl_handle_s *h, const double *x, int64_t len, bool *out)
{
    double *partials, *scalars;
    CTL_TRY(vec_workspace(h, &partials, &scalars));
    const int64_t len2 = len / 2;
    asum_kernel<<<grid_for(len2), RT, 0, h->stream>>>(x, len2, partials);
    h->launches++;
    double s = 0.0;
    CTL_TRY(sum_partials_host(h, grid_for(len2), &s));
    *out = s == 0.0;
    return CTL_OK;
}
