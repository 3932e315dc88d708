// Krylov vector primitives (vec_ops.cu).  `len` is always even (ld is a multiple of 8).
#pragma once
#include "common.cuh"

int vec_workspace(ctl_handle_s *h, double **partials, double **scalars);
int vec_zero(ctl_handle_s *h, double *x, int64_t len);
int vec_copy(ctl_handle_s *h, double *dst, const double *src, int64_t len);
// dst = a x + b y + c z (null operands are skipped), all scaled by 1 / *inv_scalar_dev if given
int vec_lincomb(ctl_handle_s *h, double *dst, double a, const double *x, double b, const double *y,
                double c, const double *z, const double *inv_scalar_dev, int64_t len);
// out_dev[j] = V_j . w (j < k <= 64), optional square roots; results stay on the device
int vec_multi_dot_dev(ctl_handle_s *h, const double *const *V, int k, const double *w, int64_t len,
                      double *out_dev, double *out_sqrt_dev);
// w += sign * sum_j coef_dev[j] V_j, optionally followed by ||w||^2 (and its root)
int vec_maxpy_dev(ctl_handle_s *h, double *w, const double *const *V, int k, const double *coef_dev,
                  double sign, int64_t len, double *norm2_dev, double *norm_dev);
int vec_maxpy_host(ctl_handle_s *h, double *w, const double *const *V, int k, const double *coef_host,
                   double sign, int64_t len);
int vec_sqrt_dev(ctl_handle_s *h, const double *in, double *out, int k);
int vec_read_scalars(ctl_handle_s *h, const double *dev, int k, double *host_out);
int vec_dot_host(ctl_handle_s *h, const double *x, const double *y, int64_t len, double *out);
int vec_norm_host(ctl_handle_s *h, const double *x, int64_t len, double *out);

// with_internal for the heat-type handle: the caller's vectors are block-major, or time-fastest (copied)
template <size_t K, class F>
int with_tf(ctl_handle_s *h, int layout, const double *const (&in)[K], double *out, F fn)
{
    const bool tf = layout == CTL_LAYOUT_TIME_FASTEST;
    const int64_t len = h->vec_len();
    return with_internal(
        h->pool, in, out,
        [&](const double *src, double *dst) { return tf ? vec_copy(h, dst, src, len) : ctl_to_tf(h, src, dst); },
        [&](const double *src, double *dst) { return tf ? vec_copy(h, dst, src, len) : ctl_to_bm(h, src, dst); }, fn);
}
