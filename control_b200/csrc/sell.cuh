// Single-column sparse products of the time sweeps and AMG cycles (SURVEY.md rows K8, K9): matrices, formats
// and the kernel entry points (sell.cu).
//
// Every product inside the sweeps acts on ONE spatial vector, so rows cannot be spread over a warp the way the
// time-batched kernels do.  Two layouts:
//   SELL-32      one thread per row, coalesced stream loads (mesh stencils, the large Galerkin levels);
//   CSR-vector   `lanes` threads per row with a shuffle reduction (long rows: restrictions, small coarse levels).
// Both come in the exact compressed formats of sell_format.h.  A matrix remembers the exchange plan of its gathered
// vector (multi-GPU, halo.cuh): kernels wait for the ghost values they gather and push the boundary rows they produce
// straight into the neighbours' memory.
#pragma once
#include <memory>

#include "common.cuh"
#include "halo.cuh"
#include "sell_format.h"

struct SellPattern {
    int n_rows = 0, n_cols = 0, n_slices = 0;
    int64_t n_stored = 0, nnz = 0;
    int2 *sp = nullptr;                // device, n_slices + 1: (first stored position, column base)
    int *cols = nullptr;               // device, n_stored
    uint16_t *dcol = nullptr;          // device, n_stored (null: 16-bit offsets not available)
    SfSellLayout host;                 // kept: value sets are laid out on it later (sell_set_values)
    ~SellPattern();
};

struct SellMat {
    std::shared_ptr<SellPattern> pat;
    int fmt = FMT_F64;
    bool stream = false;               // matrix larger than the L2 share it can keep: evict-first loads
    int n_own = 0;                     // gathered columns >= n_own come from the ghost array (0: all owned)
    int nc = 1;                        // components: the scalar matrix S acts on nc interleaved vectors, dof = nc * row
                                       // + comp (I_nc (x) S, one GPU only); vectors have nc * n_rows entries
    int64_t bytes_per_pass = 0;        // matrix stream bytes of one product (byte model)
    // SELL value arrays (owned)
    double *vals = nullptr;
    uint16_t *vcode = nullptr;
    double *vdict = nullptr;
    void *code = nullptr;
    DictEnt *dict = nullptr;
    int4 *sp4 = nullptr;               // FMT_STENCIL
    DictEnt *stab = nullptr;
    int ps_off = -2, ps_w = 0;         // FMT_STENCIL: most frequent stencil (kernel-parameter copy in view())
    DictEnt ps[SF_PS];
    // CSR-vector form (lanes > 0): owns all of its arrays
    int lanes = 0;
    int *csr_ptr = nullptr, *csr_cols = nullptr, *csr_rbase = nullptr;
    uint16_t *csr_dcol = nullptr;
    double *csr_vals = nullptr;

    int n_rows() const { return pat->n_rows; }
    bool valid() const { return pat != nullptr; }
    MatView view() const;
};

// build the pattern from a host CSR (column indices need not be sorted)
int sell_build_pattern(ctl_handle_s *h, const HostCSR &A, std::shared_ptr<SellPattern> &out);
// lay one value set (CSR order, host) out on a pattern, in the most compact exact format
int sell_set_values(ctl_handle_s *h, const std::shared_ptr<SellPattern> &pat, const double *csr_values, SellMat &out);
// one call for matrices that own their pattern: picks SELL or CSR-vector by mean row length
// (force_lanes > 0: CSR-vector with that many lanes per row)
int sell_from_csr(ctl_handle_s *h, const HostCSR &A, SellMat &out, int force_lanes = 0);
void sell_free(SellMat &m);

enum SellMode {
    SELL_ASSIGN = 0,      // y  = A x
    SELL_RESIDUAL = 1,    // y  = b - A x
    SELL_ADD = 2,         // y += A x
    SELL_SUB = 3,         // y -= A x
    SELL_BPLUS = 4        // y  = b + A x
};

// A gathered vector: owned entries and (multi-GPU) its ghost entries, either stored plainly (completed earlier) or
// still in the slot of the exchange that delivers them (`ll`, with the exchange's index + 1: the gathering kernel
// spins on the entries it reads, halo.cuh).
struct GVec {
    const double *x = nullptr;
    const double *ghost = nullptr;
    const ulonglong2 *ll = nullptr;
    unsigned idx1 = 0;
    GVec() {}
    GVec(const double *x_) : x(x_) {}
    GVec(const double *x_, const double *g_) : x(x_), ghost(g_) {}
    GVec(const double *x_, const ulonglong2 *ll_, unsigned idx1_) : x(x_), ll(ll_), idx1(idx1_) {}
};

int sell_spmv(ctl_handle_s *h, const SellMat &A, const GVec &x, double *y, const double *b, int mode,
              const HaloPush &push = HaloPush());
// Chebyshev / Jacobi step: out = a * p_prev + bq * p_cur + c * dinv .* (b - A p_cur)
// (p_prev may be null when a == 0; out may alias p_prev).  prev_scale != 0: p_prev is not read but taken as
// prev_scale * dinv .* b (the first iterate from a zero guess, never stored).
int sell_cheb_step(ctl_handle_s *h, const SellMat &A, const double *dinv, const double *b, const double *p_prev,
                   const GVec &p_cur, double *out, double a, double bq, double c, double prev_scale = 0.0,
                   const HaloPush &push = HaloPush());
// the first TWO steps from a zero guess in one kernel: p1 = s dinv .* b is formed on the fly at the gathered
// columns, out = w p1 + w s dinv .* (b - A p1)   (dinv and b are gathered: both need their ghost entries)
int sell_cheb_first2(ctl_handle_s *h, const SellMat &A, const GVec &dinv, const GVec &b, double *out, double s, double w,
                     const HaloPush &push = HaloPush());
// out = c * dinv .* b   (first step from a zero guess); n rows of nc interleaved components, dinv per row
int vec_dinv_scale(ctl_handle_s *h, const double *dinv, const double *b, double *out, double c, int n,
                   const HaloPush &push = HaloPush(), int nc = 1);
// y = Ainv b, dense row-major n x n with row stride lda (even); b and y hold nc interleaved components per row
int dense_gemv(ctl_handle_s *h, const double *Ainv, const double *b, double *y, int n, int lda, int nc = 1);
// two-matrix product on one shared row set (backward-sweep right-hand side, pc.cu):
//   y = alpha * A1 (x1 + x2) + beta * A2 x3      (x2, x3 may be null)
int sell_spmv2(ctl_handle_s *h, const SellMat &A1, const SellMat &A2, const GVec &x1, const GVec &x2, const GVec &x3,
               double *y, double alpha, double beta, const HaloPush &push = HaloPush());
int vec_copy_n(ctl_handle_s *h, double *dst, const double *src, int n);
