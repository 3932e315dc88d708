// Fused all-at-once KKT operator apply (SURVEY.md rows K1 + K2 + K3).
//
// Replaces MultiBlockSystemMatrix.mult (preconditioner/preconditioner.py:375-543): the
// 8N-4 (CN) / 6N-4 (BE) MatMultAdd calls over separately assembled blocks
// (control/control.py:2889-2978), the T_1 / T_2 time-coupling transforms (437-470) and the
// DirichletBCNullspace pre/post corrections (384-393, 527-537) become ONE kernel:
//
//   * vectors live in the time-fastest layout X[row][ld]: the N time columns of a spatial
//     dof are contiguous, so a (sub-)warp reads the whole N-column row segment of a
//     gathered dof with coalesced 16-byte loads (lane l owns columns 2l, 2l+1);
//   * every time step shares the pattern and the values of M and K, so the matrix is read
//     once per row, not once per block (per-level values: [nnz][ld] panels, same access);
//   * the four products MV, KV, MZ, KZ of a row stay in registers; the block stencil and
//     T_1 / T_2 are neighbour exchanges along the time axis = warp shuffles;
//   * Dirichlet columns are eliminated from the value arrays at setup (x_c = P x) and
//     Dirichlet rows return x (y = P A P x + (I - P) x).
//
// HBM-bound: algorithmic bytes per apply = 32 n N + 20 nnz + 4 (n+1) (BASELINE.md section 3).
#include <algorithm>

#include "common.cuh"

namespace {

constexpr int STAGE_CAP = 1024;   // CSR entries a CTA stages in shared memory
constexpr int CHUNK = 8;
#ifndef SCHUNK
#define SCHUNK 4
#endif
#ifndef SMINB
#define SMINB 4
#endif          // matrix entries staged per pass (covers a P1 2-D row)

struct KktArgs {
    int n_rows;                   // owned rows
    int n_own_cols;               // columns < n_own_cols come from x, the rest from halo
    int N, ld;
    const int *indptr, *indices;
    const double *Mv, *Kv, *KTv;  // value sets (BC columns zeroed)
    const uint8_t *bcmask;
    const double *xv, *xz;        // input panels  [n_rows x ld]
    const double *hv, *hz;        // ghost rows    [n_halo x ld]
    double *y0, *y1;              // output panels
    double tau, beta;
};

__device__ __forceinline__ double2 ldg2(const double *p)
{
    return __ldg(reinterpret_cast<const double2 *>(p));
}

// G = lanes per row (ld = 2 G columns); 32 / G rows per warp.
template <bool CN, bool PER_LEVEL, int G>
__global__ void __launch_bounds__(256) kkt_apply_kernel(const KktArgs a)
{
    constexpr int ROWS_PER_WARP = 32 / G;
    const int lane = threadIdx.x & 31;
    const int sub = lane / G;
    const int l = lane % G;
    const int warp = (blockIdx.x * (blockDim.x >> 5)) + (threadIdx.x >> 5);
    const int row = warp * ROWS_PER_WARP + sub;
    const bool live = row < a.n_rows;
    const int r = live ? row : a.n_rows - 1;        // keep the whole warp in the shuffles
    const int c0 = 2 * l;
    const int ld = a.ld;

    double mv0 = 0, mv1 = 0, kv0 = 0, kv1 = 0, mz0 = 0, mz1 = 0, kz0 = 0, kz1 = 0;

    const int kbeg = a.indptr[r], kend = a.indptr[r + 1];
    for (int k0 = kbeg; k0 < kend; k0 += CHUNK) {
        int col[CHUNK];
        double m[CHUNK];
#pragma unroll
        for (int j = 0; j < CHUNK; ++j) {
            const int k = k0 + j;
            const bool ok = k < kend;
            col[j] = ok ? __ldg(a.indices + k) : r;
            m[j] = ok ? __ldg(a.Mv + k) : 0.0;
        }
        double2 xv[CHUNK], xz[CHUNK];
#pragma unroll
        for (int j = 0; j < CHUNK; ++j) {
            const int c = col[j];
            const bool own = c < a.n_own_cols;
            const double *pv = own ? a.xv + (size_t)c * ld : a.hv + (size_t)(c - a.n_own_cols) * ld;
            const double *pz = own ? a.xz + (size_t)c * ld : a.hz + (size_t)(c - a.n_own_cols) * ld;
            xv[j] = ldg2(pv + c0);
            xz[j] = ldg2(pz + c0);
        }
        if (!PER_LEVEL) {
            double kk[CHUNK], kt[CHUNK];
#pragma unroll
            for (int j = 0; j < CHUNK; ++j) {
                const int k = k0 + j;
                const bool ok = k < kend;
                kk[j] = ok ? __ldg(a.Kv + k) : 0.0;
                kt[j] = ok ? __ldg(a.KTv + k) : 0.0;
            }
#pragma unroll
            for (int j = 0; j < CHUNK; ++j) {
                mv0 = fma(m[j], xv[j].x, mv0);
                mv1 = fma(m[j], xv[j].y, mv1);
                mz0 = fma(m[j], xz[j].x, mz0);
                mz1 = fma(m[j], xz[j].y, mz1);
                kv0 = fma(kk[j], xv[j].x, kv0);
                kv1 = fma(kk[j], xv[j].y, kv1);
                kz0 = fma(kt[j], xz[j].x, kz0);
                kz1 = fma(kt[j], xz[j].y, kz1);
            }
        } else {
#pragma unroll
            for (int j = 0; j < CHUNK; ++j) {
                const int k = k0 + j;
                if (k < kend) {
                    const double2 kk = ldg2(a.Kv + (size_t)k * ld + c0);
                    const double2 kt = ldg2(a.KTv + (size_t)k * ld + c0);
                    mv0 = fma(m[j], xv[j].x, mv0);
                    mv1 = fma(m[j], xv[j].y, mv1);
                    mz0 = fma(m[j], xz[j].x, mz0);
                    mz1 = fma(m[j], xz[j].y, mz1);
                    kv0 = fma(kk.x, xv[j].x, kv0);
                    kv1 = fma(kk.y, xv[j].y, kv1);
                    kz0 = fma(kt.x, xz[j].x, kz0);
                    kz1 = fma(kt.y, xz[j].y, kz1);
                }
            }
        }
    }

    // ---- block stencil + T_1 / T_2 along the time axis (columns c0, c0+1 of this lane)
    const unsigned full = 0xffffffffu;
    const bool first = (l == 0), last = (l == G - 1);
    const int N = a.N;
    const bool in0 = c0 < N, in1 = c0 + 1 < N;
    double y00, y01, y10, y11;
    if (CN) {
        const double h = 0.5 * a.tau, hb = h / a.beta;
        double t;
        t = __shfl_up_sync(full, mv1, 1, G);   const double mvp0 = first ? 0.0 : t;
        t = __shfl_up_sync(full, kv1, 1, G);   const double kvp0 = first ? 0.0 : t;
        t = __shfl_down_sync(full, kz0, 1, G); const double kzn1 = last ? 0.0 : t;
        t = __shfl_down_sync(full, mz0, 1, G); const double mzn1 = last ? 0.0 : t;
        // rows of the untransformed block system (control/control.py:2938-2958)
        double r00 = h * (mvp0 + mv0) + h * (kz0 + kz1) + mz0 - mz1;
        double r01 = h * (mv0 + mv1) + h * (kz1 + kzn1) + mz1 - mzn1;
        double r10 = h * (kvp0 + kv0) - mvp0 + mv0 - hb * (mz0 + mz1);
        double r11 = h * (kv0 + kv1) - mv0 + mv1 - hb * (mz1 + mzn1);
        if (!in0) { r00 = 0.0; r10 = 0.0; }
        if (!in1) { r01 = 0.0; r11 = 0.0; }
        // T_1: add the next block row; T_2: add the previous one (preconditioner.py:33-60)
        t = __shfl_down_sync(full, r00, 1, G); const double r0n = last ? 0.0 : t;
        t = __shfl_up_sync(full, r11, 1, G);   const double r1p = first ? 0.0 : t;
        y00 = r00 + r01;
        y01 = r01 + r0n;
        y10 = r10 + r1p;
        y11 = r11 + r10;
    } else {
        const double tau = a.tau, tb = tau / a.beta;
        double t;
        t = __shfl_up_sync(full, mv1, 1, G);   const double mvp0 = first ? 0.0 : t;
        t = __shfl_down_sync(full, mz0, 1, G); const double mzn1 = last ? 0.0 : t;
        // control/control.py:2907-2928, 2960-2978: block_00 last row None, block_11 row 0 None
        y00 = tau * kz0 + mz0 + ((c0 < N - 1) ? (tau * mv0 - mz1) : 0.0);
        y01 = tau * kz1 + mz1 + ((c0 + 1 < N - 1) ? (tau * mv1 - mzn1) : 0.0);
        y10 = tau * kv0 + mv0 + ((c0 >= 1) ? (-mvp0 - tb * mz0) : 0.0);
        y11 = tau * kv1 + mv1 + (-mv0 - tb * mz1);
    }
    if (!in0) { y00 = 0.0; y10 = 0.0; }
    if (!in1) { y01 = 0.0; y11 = 0.0; }
    if (!live) return;
    if (a.bcmask[r]) {           // y = (I - P) x on constrained rows
        const double2 xv = ldg2(a.xv + (size_t)r * ld + c0);
        const double2 xz = ldg2(a.xz + (size_t)r * ld + c0);
        y00 = xv.x; y01 = xv.y; y10 = xz.x; y11 = xz.y;
    }
    *reinterpret_cast<double2 *>(a.y0 + (size_t)r * ld + c0) = make_double2(y00, y01);
    *reinterpret_cast<double2 *>(a.y1 + (size_t)r * ld + c0) = make_double2(y10, y11);
}


// ---------------------------------------------------------------------------------------
// Staged variant (the one normally launched): a CTA owns `rows_per_cta` consecutive rows.
// Their CSR entries are contiguous, so the CTA first copies them into shared memory with
// fully coalesced loads, already converted to what the inner loop needs: the BYTE offset of
// the gathered X row (32 bit) and the (M, K) value pair as one 16-byte word.  Afterwards the
// only global latency a warp sees per row is the gather of the X row segments themselves.
// History (profiles/): v1 unstaged = latency bound (1.51 ms); v2 staged = 0.74 ms but issue
// bound (67% issue slots, 574 M warp instructions of which 11% DFMA: address IMADs, constant
// reloads, predication selects); v3 below cuts the per-entry overhead to two LDS, one
// integer add, two LDG.128 and eight DFMA.
// ---------------------------------------------------------------------------------------
template <bool CN, bool PER_LEVEL, bool SYM, bool HALO, int G, int SC>
__global__ void __launch_bounds__(256, SMINB) kkt_apply_staged_kernel(const KktArgs a, const int rows_per_cta,
                                                                     const int cap)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // layout: [cap+1] double2 (m, k) | [cap+1] double kt (only !SYM) | [cap+1] unsigned off | [rows+1] int ptr
    double2 *s_mk = reinterpret_cast<double2 *>(smem_raw);
    double *s_kt = reinterpret_cast<double *>(s_mk + (cap + 1));
    unsigned *s_off = reinterpret_cast<unsigned *>(SYM || PER_LEVEL ? s_kt : s_kt + (cap + 1));
    int *s_ptr = reinterpret_cast<int *>(s_off + (cap + 1));

    constexpr int RPW = 32 / G;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int sub = lane / G, l = lane % G;
    const int c0 = 2 * l;
    const int ld = a.ld;
    const int r0 = blockIdx.x * rows_per_cta;
    const int nrows = min(rows_per_cta, a.n_rows - r0);
    const int n_own = a.n_own_cols;
    const char *__restrict__ xv_b = reinterpret_cast<const char *>(a.xv);
    const char *__restrict__ xz_b = reinterpret_cast<const char *>(a.xz);
    const char *__restrict__ hv_b = reinterpret_cast<const char *>(a.hv);
    const char *__restrict__ hz_b = reinterpret_cast<const char *>(a.hz);
    const unsigned lane_b = (unsigned)c0 * 8u;
    const unsigned row_b = (unsigned)ld * 8u;

    for (int i = threadIdx.x; i <= nrows; i += blockDim.x) s_ptr[i] = __ldg(a.indptr + r0 + i);
    __syncthreads();
    const int kb = s_ptr[0];
    const int cnt = s_ptr[nrows] - kb;
    for (int k = threadIdx.x; k < cnt; k += blockDim.x) {
        const int c = __ldg(a.indices + kb + k);
        // ghost rows (HALO) are addressed relative to the halo buffers: flag them in bit 31
        s_off[k] = (HALO && c >= n_own) ? (0x80000000u | ((unsigned)(c - n_own) * row_b)) : (unsigned)c * row_b;
        s_mk[k] = make_double2(__ldg(a.Mv + kb + k), PER_LEVEL ? 0.0 : __ldg(a.Kv + kb + k));
        if (!PER_LEVEL && !SYM) s_kt[k] = __ldg(a.KTv + kb + k);
    }
    if (threadIdx.x == 0) {          // sentinel entry: zero values, a valid row to gather
        s_off[cap] = 0u;
        s_mk[cap] = make_double2(0.0, 0.0);
        if (!PER_LEVEL && !SYM) s_kt[cap] = 0.0;
    }
    __syncthreads();

    const unsigned full = 0xffffffffu;
    const bool first = (l == 0), last = (l == G - 1);
    const int N = a.N;
    const bool in0 = c0 < N, in1 = c0 + 1 < N;
    const double tau = a.tau, beta = a.beta;
    const int nwarps = blockDim.x >> 5;

    for (int base = wid * RPW; base < nrows; base += nwarps * RPW) {
        const int lr_raw = base + sub;
        const bool live = lr_raw < nrows;
        const int lr = live ? lr_raw : nrows - 1;
        const int r = r0 + lr;
        const int kbeg = s_ptr[lr] - kb, kend = s_ptr[lr + 1] - kb;
        double mv0 = 0, mv1 = 0, kv0 = 0, kv1 = 0, mz0 = 0, mz1 = 0, kz0 = 0, kz1 = 0;
        for (int k0 = kbeg; k0 < kend; k0 += SC) {
            unsigned off[SC];
            int kk[SC];
#pragma unroll
            for (int j = 0; j < SC; ++j) {
                kk[j] = (k0 + j < kend) ? k0 + j : cap;       // padding slots read the sentinel
                off[j] = s_off[kk[j]];
            }
            double2 xv[SC], xz[SC];
#pragma unroll
            for (int j = 0; j < SC; ++j) {
                if (HALO && (off[j] & 0x80000000u)) {
                    const unsigned o = (off[j] & 0x7fffffffu) + lane_b;
                    xv[j] = __ldg(reinterpret_cast<const double2 *>(hv_b + o));
                    xz[j] = __ldg(reinterpret_cast<const double2 *>(hz_b + o));
                } else {
                    const unsigned o = off[j] + lane_b;
                    xv[j] = __ldg(reinterpret_cast<const double2 *>(xv_b + o));
                    xz[j] = __ldg(reinterpret_cast<const double2 *>(xz_b + o));
                }
            }
#pragma unroll
            for (int j = 0; j < SC; ++j) {
                const double2 mk = s_mk[kk[j]];
                mv0 = fma(mk.x, xv[j].x, mv0);
                mv1 = fma(mk.x, xv[j].y, mv1);
                mz0 = fma(mk.x, xz[j].x, mz0);
                mz1 = fma(mk.x, xz[j].y, mz1);
                if (!PER_LEVEL) {
                    const double kt = SYM ? mk.y : s_kt[kk[j]];
                    kv0 = fma(mk.y, xv[j].x, kv0);
                    kv1 = fma(mk.y, xv[j].y, kv1);
                    kz0 = fma(kt, xz[j].x, kz0);
                    kz1 = fma(kt, xz[j].y, kz1);
                } else if (kk[j] != cap) {
                    const double2 kp = ldg2(a.Kv + (size_t)(kb + kk[j]) * ld + c0);
                    const double2 kt = ldg2(a.KTv + (size_t)(kb + kk[j]) * ld + c0);
                    kv0 = fma(kp.x, xv[j].x, kv0);
                    kv1 = fma(kp.y, xv[j].y, kv1);
                    kz0 = fma(kt.x, xz[j].x, kz0);
                    kz1 = fma(kt.y, xz[j].y, kz1);
                }
            }
        }
        double y00, y01, y10, y11;
        if (CN) {
            const double h = 0.5 * tau, hb = h / beta;
            double t;
            t = __shfl_up_sync(full, mv1, 1, G);   const double mvp0 = first ? 0.0 : t;
            t = __shfl_up_sync(full, kv1, 1, G);   const double kvp0 = first ? 0.0 : t;
            t = __shfl_down_sync(full, kz0, 1, G); const double kzn1 = last ? 0.0 : t;
            t = __shfl_down_sync(full, mz0, 1, G); const double mzn1 = last ? 0.0 : t;
            double r00 = h * (mvp0 + mv0) + h * (kz0 + kz1) + mz0 - mz1;
            double r01 = h * (mv0 + mv1) + h * (kz1 + kzn1) + mz1 - mzn1;
            double r10 = h * (kvp0 + kv0) - mvp0 + mv0 - hb * (mz0 + mz1);
            double r11 = h * (kv0 + kv1) - mv0 + mv1 - hb * (mz1 + mzn1);
            if (!in0) { r00 = 0.0; r10 = 0.0; }
            if (!in1) { r01 = 0.0; r11 = 0.0; }
            t = __shfl_down_sync(full, r00, 1, G); const double r0n = last ? 0.0 : t;
            t = __shfl_up_sync(full, r11, 1, G);   const double r1p = first ? 0.0 : t;
            y00 = r00 + r01;
            y01 = r01 + r0n;
            y10 = r10 + r1p;
            y11 = r11 + r10;
        } else {
            const double tb = tau / beta;
            double t;
            t = __shfl_up_sync(full, mv1, 1, G);   const double mvp0 = first ? 0.0 : t;
            t = __shfl_down_sync(full, mz0, 1, G); const double mzn1 = last ? 0.0 : t;
            y00 = tau * kz0 + mz0 + ((c0 < N - 1) ? (tau * mv0 - mz1) : 0.0);
            y01 = tau * kz1 + mz1 + ((c0 + 1 < N - 1) ? (tau * mv1 - mzn1) : 0.0);
            y10 = tau * kv0 + mv0 + ((c0 >= 1) ? (-mvp0 - tb * mz0) : 0.0);
            y11 = tau * kv1 + mv1 + (-mv0 - tb * mz1);
        }
        if (!in0) { y00 = 0.0; y10 = 0.0; }
        if (!in1) { y01 = 0.0; y11 = 0.0; }
        if (live) {
            const size_t ro = (size_t)r * ld + c0;
            if (a.bcmask[r]) {
                const double2 xv = ldg2(a.xv + ro);
                const double2 xz = ldg2(a.xz + ro);
                y00 = xv.x; y01 = xv.y; y10 = xz.x; y11 = xz.y;
            }
            // streaming stores: the 1 GB result must not push the X rows still to be gathered out of L2
            __stcs(reinterpret_cast<double2 *>(a.y0 + ro), make_double2(y00, y01));
            __stcs(reinterpret_cast<double2 *>(a.y1 + ro), make_double2(y10, y11));
        }
    }
}

template <bool CN, bool PER_LEVEL, bool SYM, bool HALO>
void launch_staged_h(const KktArgs &a, int G, int rows_per_cta, int cap, int chunk, cudaStream_t s)
{
    const int blocks = ceil_div(a.n_rows, rows_per_cta);
    const size_t smem = (size_t)(cap + 1) * (16 + ((SYM || PER_LEVEL) ? 0 : 8) + 4) + (size_t)(rows_per_cta + 1) * 4;
#define LS(GG, CC) kkt_apply_staged_kernel<CN, PER_LEVEL, SYM, HALO, GG, CC><<<blocks, 256, smem, s>>>(a, rows_per_cta, cap)
    if (G == 32 && !PER_LEVEL) {
        // chunk = entries gathered per pass; matched to the row length so that no padding
        // slots are processed (7 for a P1 triangle mesh, 5 for the 15-point P1 tetrahedra stencil)
        switch (chunk) {
        case 5: LS(32, 5); break;
        case 7: LS(32, 7); break;
        case 8: LS(32, 8); break;
        default: LS(32, 4); break;
        }
        return;
    }
    switch (G) {
    case 4: LS(4, 4); break;
    case 8: LS(8, 4); break;
    case 16: LS(16, 4); break;
    default: LS(32, 4); break;
    }
#undef LS
}

template <bool CN, bool PER_LEVEL, bool SYM>
void launch_staged(const KktArgs &a, int G, int rows_per_cta, int cap, int chunk, bool halo, cudaStream_t s)
{
    if (halo) launch_staged_h<CN, PER_LEVEL, SYM, true>(a, G, rows_per_cta, cap, chunk, s);
    else launch_staged_h<CN, PER_LEVEL, SYM, false>(a, G, rows_per_cta, cap, chunk, s);
}

// ---------------------------------------------------------------------------------------
// Wide variant for more than 64 time blocks (ld = 128 or 256): one warp per row, every lane
// owns CPL = ld / 32 CONSECUTIVE time columns, so the block stencil and T_1 / T_2 only cross
// lanes at the ends of a lane's column group.  Same staging as the kernel above.
// ---------------------------------------------------------------------------------------
template <int CPL>
__device__ __forceinline__ void time_prev(const double (&a)[CPL], double (&out)[CPL], int lane)
{
    const double t = __shfl_up_sync(0xffffffffu, a[CPL - 1], 1);
    out[0] = lane == 0 ? 0.0 : t;
#pragma unroll
    for (int c = 1; c < CPL; ++c) out[c] = a[c - 1];
}

template <int CPL>
__device__ __forceinline__ void time_next(const double (&a)[CPL], double (&out)[CPL], int lane)
{
    const double t = __shfl_down_sync(0xffffffffu, a[0], 1);
#pragma unroll
    for (int c = 0; c < CPL - 1; ++c) out[c] = a[c + 1];
    out[CPL - 1] = lane == 31 ? 0.0 : t;
}

template <bool CN, bool PER_LEVEL, bool SYM, bool HALO, int CPL>
__global__ void __launch_bounds__(256) kkt_apply_wide_kernel(const KktArgs a, const int rows_per_cta, const int cap)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2 *s_mk = reinterpret_cast<double2 *>(smem_raw);
    double *s_kt = reinterpret_cast<double *>(s_mk + (cap + 1));
    int *s_col = reinterpret_cast<int *>(SYM || PER_LEVEL ? s_kt : s_kt + (cap + 1));
    int *s_ptr = s_col + (cap + 1);

    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int c0 = CPL * lane;
    const int ld = a.ld;
    const int r0 = blockIdx.x * rows_per_cta;
    const int nrows = min(rows_per_cta, a.n_rows - r0);

    for (int i = threadIdx.x; i <= nrows; i += blockDim.x) s_ptr[i] = __ldg(a.indptr + r0 + i);
    __syncthreads();
    const int kb = s_ptr[0];
    const int cnt = s_ptr[nrows] - kb;
    for (int k = threadIdx.x; k < cnt; k += blockDim.x) {
        s_col[k] = __ldg(a.indices + kb + k);
        s_mk[k] = make_double2(__ldg(a.Mv + kb + k), PER_LEVEL ? 0.0 : __ldg(a.Kv + kb + k));
        if (!PER_LEVEL && !SYM) s_kt[k] = __ldg(a.KTv + kb + k);
    }
    __syncthreads();

    const int N = a.N;
    const double tau = a.tau, beta = a.beta;
    for (int lr = wid; lr < nrows; lr += (blockDim.x >> 5)) {
        const int r = r0 + lr;
        const int kbeg = s_ptr[lr] - kb, kend = s_ptr[lr + 1] - kb;
        double mv[CPL], kv[CPL], mz[CPL], kz[CPL];
#pragma unroll
        for (int c = 0; c < CPL; ++c) mv[c] = kv[c] = mz[c] = kz[c] = 0.0;
        for (int k = kbeg; k < kend; ++k) {
            const int col = s_col[k];
            const bool own = !HALO || col < a.n_own_cols;
            const double *pv = own ? a.xv + (size_t)col * ld : a.hv + (size_t)(col - a.n_own_cols) * ld;
            const double *pz = own ? a.xz + (size_t)col * ld : a.hz + (size_t)(col - a.n_own_cols) * ld;
            const double2 mk = s_mk[k];
            const double kt = (SYM || PER_LEVEL) ? mk.y : s_kt[k];
#pragma unroll
            for (int q = 0; q < CPL / 2; ++q) {
                const double2 xv = ldg2(pv + c0 + 2 * q);
                const double2 xz = ldg2(pz + c0 + 2 * q);
                double2 kk = make_double2(mk.y, mk.y), kkt = make_double2(kt, kt);
                if (PER_LEVEL) {
                    kk = ldg2(a.Kv + (size_t)(kb + k) * ld + c0 + 2 * q);
                    kkt = ldg2(a.KTv + (size_t)(kb + k) * ld + c0 + 2 * q);
                }
                mv[2 * q] = fma(mk.x, xv.x, mv[2 * q]);
                mv[2 * q + 1] = fma(mk.x, xv.y, mv[2 * q + 1]);
                mz[2 * q] = fma(mk.x, xz.x, mz[2 * q]);
                mz[2 * q + 1] = fma(mk.x, xz.y, mz[2 * q + 1]);
                kv[2 * q] = fma(kk.x, xv.x, kv[2 * q]);
                kv[2 * q + 1] = fma(kk.y, xv.y, kv[2 * q + 1]);
                kz[2 * q] = fma(kkt.x, xz.x, kz[2 * q]);
                kz[2 * q + 1] = fma(kkt.y, xz.y, kz[2 * q + 1]);
            }
        }
        double y0[CPL], y1[CPL];
        if (CN) {
            const double h = 0.5 * tau, hb = h / beta;
            double mvp[CPL], kvp[CPL], kzn[CPL], mzn[CPL], r0v[CPL], r1v[CPL], r0n[CPL], r1p[CPL];
            time_prev<CPL>(mv, mvp, lane);
            time_prev<CPL>(kv, kvp, lane);
            time_next<CPL>(kz, kzn, lane);
            time_next<CPL>(mz, mzn, lane);
#pragma unroll
            for (int c = 0; c < CPL; ++c) {
                const bool in = c0 + c < N;
                r0v[c] = in ? h * (mvp[c] + mv[c]) + h * (kz[c] + kzn[c]) + mz[c] - mzn[c] : 0.0;
                r1v[c] = in ? h * (kvp[c] + kv[c]) - mvp[c] + mv[c] - hb * (mz[c] + mzn[c]) : 0.0;
            }
            time_next<CPL>(r0v, r0n, lane);
            time_prev<CPL>(r1v, r1p, lane);
#pragma unroll
            for (int c = 0; c < CPL; ++c) {
                y0[c] = r0v[c] + r0n[c];
                y1[c] = r1v[c] + r1p[c];
            }
        } else {
            const double tb = tau / beta;
            double mvp[CPL], mzn[CPL];
            time_prev<CPL>(mv, mvp, lane);
            time_next<CPL>(mz, mzn, lane);
#pragma unroll
            for (int c = 0; c < CPL; ++c) {
                const int col = c0 + c;
                y0[c] = tau * kz[c] + mz[c] + ((col < N - 1) ? (tau * mv[c] - mzn[c]) : 0.0);
                y1[c] = tau * kv[c] + mv[c] + ((col >= 1) ? (-mvp[c] - tb * mz[c]) : 0.0);
            }
        }
        const size_t ro = (size_t)r * ld + c0;
        const bool bc = a.bcmask[r] != 0;
#pragma unroll
        for (int q = 0; q < CPL / 2; ++q) {
            double2 o0 = make_double2(c0 + 2 * q < N ? y0[2 * q] : 0.0, c0 + 2 * q + 1 < N ? y0[2 * q + 1] : 0.0);
            double2 o1 = make_double2(c0 + 2 * q < N ? y1[2 * q] : 0.0, c0 + 2 * q + 1 < N ? y1[2 * q + 1] : 0.0);
            if (bc) {
                o0 = ldg2(a.xv + ro + 2 * q);
                o1 = ldg2(a.xz + ro + 2 * q);
            }
            __stcs(reinterpret_cast<double2 *>(a.y0 + ro + 2 * q), o0);
            __stcs(reinterpret_cast<double2 *>(a.y1 + ro + 2 * q), o1);
        }
    }
}

template <bool CN, bool PER_LEVEL, bool SYM, bool HALO>
void launch_wide_h(const KktArgs &a, int rows_per_cta, int cap, cudaStream_t s)
{
    const int blocks = ceil_div(a.n_rows, rows_per_cta);
    const size_t smem = (size_t)(cap + 1) * (16 + ((SYM || PER_LEVEL) ? 0 : 8) + 4) + (size_t)(rows_per_cta + 1) * 4;
    if (a.ld == 128) kkt_apply_wide_kernel<CN, PER_LEVEL, SYM, HALO, 4><<<blocks, 256, smem, s>>>(a, rows_per_cta, cap);
    else kkt_apply_wide_kernel<CN, PER_LEVEL, SYM, HALO, 8><<<blocks, 256, smem, s>>>(a, rows_per_cta, cap);
}

template <bool CN>
void launch_wide(const KktArgs &a, bool per_level, bool sym, bool halo, int rows_per_cta, int cap, cudaStream_t s)
{
    if (per_level) {
        if (halo) launch_wide_h<CN, true, false, true>(a, rows_per_cta, cap, s);
        else launch_wide_h<CN, true, false, false>(a, rows_per_cta, cap, s);
    } else if (sym) {
        if (halo) launch_wide_h<CN, false, true, true>(a, rows_per_cta, cap, s);
        else launch_wide_h<CN, false, true, false>(a, rows_per_cta, cap, s);
    } else {
        if (halo) launch_wide_h<CN, false, false, true>(a, rows_per_cta, cap, s);
        else launch_wide_h<CN, false, false, false>(a, rows_per_cta, cap, s);
    }
}

template <bool CN, bool PER_LEVEL>
void launch_g(const KktArgs &a, int G, cudaStream_t s)
{
    const int threads = 256;
    const int rows_per_block = (threads / 32) * (32 / G);
    const int blocks = ceil_div(a.n_rows, rows_per_block);
    switch (G) {
    case 4: kkt_apply_kernel<CN, PER_LEVEL, 4><<<blocks, threads, 0, s>>>(a); break;
    case 8: kkt_apply_kernel<CN, PER_LEVEL, 8><<<blocks, threads, 0, s>>>(a); break;
    case 16: kkt_apply_kernel<CN, PER_LEVEL, 16><<<blocks, threads, 0, s>>>(a); break;
    default: kkt_apply_kernel<CN, PER_LEVEL, 32><<<blocks, threads, 0, s>>>(a); break;
    }
}

}  // namespace

int ctl_kkt_apply_tf(ctl_handle_s *h, const double *x_tf, double *y_tf)
{
    CTL_CHECK(h->assembled, CTL_ERR_STATE, "ctl_kkt_apply: ctl_assemble has not been called");
    CTL_CHECK(h->cfg.world == 1 || h->comm, CTL_ERR_STATE, "ctl_kkt_apply: call ctl_comm_init first (world > 1)");
    if (h->n_halo > 0) CTL_TRY(ctl_halo_exchange(h, x_tf));
    KktArgs a;
    a.n_rows = h->n_loc;
    a.n_own_cols = h->n_loc;
    a.N = h->N;
    a.ld = h->ld;
    a.indptr = h->d_indptr;
    a.indices = h->d_indices;
    a.Mv = h->d_M;
    a.Kv = h->d_K;
    a.KTv = h->d_KT;
    a.bcmask = h->d_bcmask;
    const size_t panel = (size_t)h->n_loc * h->ld;
    a.xv = x_tf;
    a.xz = x_tf + panel;
    a.hv = h->d_halo;
    a.hz = h->d_halo ? h->d_halo + (size_t)h->n_halo * h->ld : nullptr;
    a.y0 = y_tf;
    a.y1 = y_tf + panel;
    a.tau = h->cfg.tau;
    a.beta = h->cfg.beta;
    const int G = h->ld / 2;
    // rows per CTA: as many consecutive rows as fit the shared-memory entry budget
    const int max_len = std::max(1, h->max_row_len);
    int rows_per_cta = std::min(64, (STAGE_CAP / max_len) / 8 * 8);
    // the staged kernel addresses gathered rows with 31-bit byte offsets
    const bool fits = (size_t)std::max(h->n_loc, h->n_halo) * h->ld * 8 < 0x7fffffffull;
    const bool staged = rows_per_cta >= 8 && fits;
    const bool halo = h->n_halo > 0;
    if (h->ld > 64) {
        CTL_CHECK(rows_per_cta >= 8, CTL_ERR_ARG, "ctl_kkt_apply: rows too long for the wide (N > 64) kernel");
        const bool sym = h->d_KT == h->d_K;
        if (h->cfg.CN) launch_wide<true>(a, h->per_level, sym, halo, rows_per_cta, rows_per_cta * max_len, h->stream);
        else launch_wide<false>(a, h->per_level, sym, halo, rows_per_cta, rows_per_cta * max_len, h->stream);
        h->launches++;
        CTL_CUDA(cudaGetLastError());
        return CTL_OK;
    }
    if (staged) {
        const int cap = rows_per_cta * max_len;
        const bool sym = h->d_KT == h->d_K;
        if (h->cfg.CN) {
            if (h->per_level) launch_staged<true, true, false>(a, G, rows_per_cta, cap, h->gather_chunk, halo, h->stream);
            else if (sym) launch_staged<true, false, true>(a, G, rows_per_cta, cap, h->gather_chunk, halo, h->stream);
            else launch_staged<true, false, false>(a, G, rows_per_cta, cap, h->gather_chunk, halo, h->stream);
        } else {
            if (h->per_level) launch_staged<false, true, false>(a, G, rows_per_cta, cap, h->gather_chunk, halo, h->stream);
            else if (sym) launch_staged<false, false, true>(a, G, rows_per_cta, cap, h->gather_chunk, halo, h->stream);
            else launch_staged<false, false, false>(a, G, rows_per_cta, cap, h->gather_chunk, halo, h->stream);
        }
    } else if (h->cfg.CN) {
        if (h->per_level) launch_g<true, true>(a, G, h->stream);
        else launch_g<true, false>(a, G, h->stream);
    } else {
        if (h->per_level) launch_g<false, true>(a, G, h->stream);
        else launch_g<false, false>(a, G, h->stream);
    }
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}
