// Single-column sparse products of the time sweeps and the AMG cycles (see sell.cuh): SELL-32 kernels (one thread
// per row) and CSR-vector kernels (T lanes per row) over the exact compressed formats of sell_format.h, with the
// device-initiated halo exchange of halo.cuh folded into every kernel.  Everything here is bound by the matrix /
// vector stream (HBM, or L2 once the compressed matrix stays resident) and by launch latency on the coarse levels;
// nothing is a dense contraction.
#include <algorithm>
#include <type_traits>

#include "sell.cuh"

SellPattern::~SellPattern()
{
    cudaFree(sp);
    cudaFree(cols);
    cudaFree(dcol);
}

void sell_free(SellMat &m)
{
    cudaFree(m.vals);
    cudaFree(m.vcode);
    cudaFree(m.vdict);
    cudaFree(m.code);
    cudaFree(m.dict);
    cudaFree(m.sp4);
    cudaFree(m.stab);
    cudaFree(m.csr_ptr);
    cudaFree(m.csr_cols);
    cudaFree(m.csr_rbase);
    cudaFree(m.csr_dcol);
    cudaFree(m.csr_vals);
    m = SellMat();
}

MatView SellMat::view() const
{
    MatView v;
    v.fmt = fmt;
    v.n_rows = pat->n_rows;
    v.n_own = n_own > 0 ? n_own : pat->n_cols;
    if (lanes) {
        v.ptr = csr_ptr;
        v.rbase = csr_rbase;
        v.cols = csr_cols;
        v.dcol = csr_dcol;
        v.vals = csr_vals;
    } else {
        v.sp = pat->sp;
        v.cols = pat->cols;
        v.dcol = pat->dcol;
        v.vals = vals;
    }
    v.vcode = vcode;
    v.vdict = vdict;
    v.code = code;
    v.dict = dict;
    v.sp4 = sp4;
    v.stab = stab;
    v.ps_off = ps_off;
    v.ps_w = ps_w;
    v.ps_dmax = 0;
    v.ps_dmin = 0;
    for (int k = 0; k < ps_w && k < SF_PS; ++k) {
        v.ps_delta[k] = ps[k].delta;
        v.ps_v[k] = ps[k].v;
        v.ps_dmax = std::max(v.ps_dmax, ps[k].delta);
        v.ps_dmin = std::min(v.ps_dmin, ps[k].delta);
    }
    return v;
}

// cap of the automatic format choice for the mesh matrices (fine level, off-diagonal blocks): every exact format
constexpr int FMT_MAX_FINE = FMT_STENCIL;

// cap for the matrices that own their pattern (coarse AMG operators, transfers) while they are small enough to
// stay in L2.  Measured at C2 (round 2, profiles/r02_inner_solve_variants.txt): on the Galerkin levels and the
// transfer operators the dictionary formats cost more instructions than their bytes save (everything there is
// L2-resident and latency bound): inner solve 0.81 ms (dictionaries) / 0.73 (16-bit offsets) / 0.67 (plain)
constexpr int FMT_MAX_COARSE = FMT_F64;

// ... "small enough": a plain (12 B per entry) stream up to this size.  Larger ones (3-D: the first Galerkin level of
// C3 has 18.5 M entries, 222 MB plain) are bound by their stream and take the most compact exact format like the
// fine level.
constexpr int64_t COARSE_PLAIN_BYTES = 64ll << 20;

// matrices whose stream exceeds this many bytes are read evict-first: they cannot stay in L2 next to the
// vectors of their level, and must not flush the coarse levels out of it
constexpr int64_t STREAM_BYTES = 40ll << 20;

template <typename T>
static int upload_vec(ctl_handle_s *h, T **dst, const std::vector<T> &src)
{
    if (*dst) {
        cudaFree(*dst);
        *dst = nullptr;
    }
    if (src.empty()) return CTL_OK;
    CTL_CUDA(cudaMalloc((void **)dst, src.size() * sizeof(T)));
    CTL_CUDA(cudaMemcpyAsync(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, h->stream));
    CTL_CUDA(cudaStreamSynchronize(h->stream));
    return CTL_OK;
}

int sell_build_pattern(ctl_handle_s *h, const HostCSR &A, std::shared_ptr<SellPattern> &out)
{
    auto p = std::make_shared<SellPattern>();
    SfCsr a;
    a.n_rows = A.n_rows;
    a.n_cols = A.n_cols;
    a.indptr = A.indptr.data();
    a.indices = A.indices.data();
    sf_sell_layout(a, p->host);
    p->n_rows = A.n_rows;
    p->n_cols = A.n_cols;
    p->n_slices = p->host.n_slices;
    p->n_stored = p->host.n_stored;
    p->nnz = p->host.nnz;
    CTL_TRY(upload_vec(h, &p->sp, p->host.sp));
    CTL_TRY(upload_vec(h, &p->cols, p->host.cols));
    CTL_TRY(upload_vec(h, &p->dcol, p->host.dcol));
    out = p;
    return CTL_OK;
}

static int sell_set_values_cap(ctl_handle_s *h, const std::shared_ptr<SellPattern> &pat, const double *csr_values, SellMat &out,
                               int max_fmt);

int sell_set_values(ctl_handle_s *h, const std::shared_ptr<SellPattern> &pat, const double *csr_values, SellMat &out)
{
    return sell_set_values_cap(h, pat, csr_values, out, FMT_MAX_FINE);
}

static int sell_set_values_cap(ctl_handle_s *h, const std::shared_ptr<SellPattern> &pat, const double *csr_values, SellMat &out,
                               int max_fmt)
{
    SfSellValues V;
    sf_sell_values(pat->host, csr_values, max_fmt, V);
    out.pat = pat;
    out.fmt = V.fmt;
    out.lanes = 0;
    out.bytes_per_pass = V.bytes_per_pass;
    out.stream = V.bytes_per_pass > STREAM_BYTES;
    CTL_TRY(upload_vec(h, &out.vals, V.vals));
    CTL_TRY(upload_vec(h, &out.vcode, V.vcode));
    CTL_TRY(upload_vec(h, &out.vdict, V.vdict));
    CTL_TRY(upload_vec(h, &out.dict, V.dict));
    CTL_TRY(upload_vec(h, &out.sp4, V.sp4));
    CTL_TRY(upload_vec(h, &out.stab, V.stab));
    out.ps_off = V.ps_off;
    out.ps_w = V.ps_w;
    for (int k = 0; k < V.ps_w && k < SF_PS; ++k) out.ps[k] = V.stab[V.ps_off + k];
    if (V.fmt == FMT_DICT8) CTL_TRY(upload_vec(h, (uint8_t **)&out.code, V.code8));
    else if (V.fmt == FMT_DICT16 || V.fmt == FMT_STENCIL) CTL_TRY(upload_vec(h, (uint16_t **)&out.code, V.code16));
    return CTL_OK;
}

int sell_from_csr(ctl_handle_s *h, const HostCSR &A, SellMat &out, int force_lanes)
{
    const double mean = A.n_rows ? (double)A.nnz() / A.n_rows : 0.0;
    // SELL-32 (one row per thread, coalesced) up to a mean row length of 24: measured at C2 against the
    // CSR-vector kernels, inner solve 0.842 ms (threshold 10) -> 0.792 (14) -> 0.774 (20-24) -> 0.779 (40)
    constexpr double SELL_MAX_MEAN = 24.0;
    // ... but only for levels with enough rows to fill the GPU with one row per thread: below ~50 k rows
    // the CSR-vector kernels (several threads per row) win (19 k-row level as SELL: 0.833 ms per solve)
    constexpr int SELL_MIN_ROWS = 50000;
    const bool mesh_like = mean <= 10.0;          // fine-mesh stencils (short rows): always SELL
    // ... and so is a level with long rows once it has enough of them (3-D: the first Galerkin level of C3, 248 k rows
    // of 75 entries): one thread per row streams coalesced indices and values (16-bit offsets: 10 B per entry),
    // where the lane-per-entry CSR kernel took 91 us per product for the same 18.5 M entries
    const bool many_rows = A.n_rows >= 100000;
    const int max_fmt = 12 * A.nnz() > COARSE_PLAIN_BYTES ? FMT_MAX_FINE : FMT_MAX_COARSE;
    if (force_lanes == 0 && (mesh_like || many_rows || (mean <= SELL_MAX_MEAN && A.n_rows >= SELL_MIN_ROWS))) {
        std::shared_ptr<SellPattern> pat;
        CTL_TRY(sell_build_pattern(h, A, pat));
        return sell_set_values_cap(h, pat, A.values.data(), out, max_fmt);
    }
    auto pat = std::make_shared<SellPattern>();     // sizes only; no SELL arrays
    pat->n_rows = A.n_rows;
    pat->n_cols = A.n_cols;
    pat->nnz = A.nnz();
    out.pat = pat;
    // lanes per row: about a quarter of the mean row length.  Measured at C2 (inner solve, warm): 8 lanes
    // for the 13-entry rows of level 1 = 0.918 ms, 16 lanes = 1.189 ms, 4 lanes = 0.843 ms: the narrow
    // groups keep four times as many rows in flight, which is what these latency-bound kernels need.
    out.lanes = mean <= 16.0 ? 4 : (mean <= 48.0 ? 8 : 16);
    if (force_lanes) out.lanes = force_lanes;
    SfCsr a;
    a.n_rows = A.n_rows;
    a.n_cols = A.n_cols;
    a.indptr = A.indptr.data();
    a.indices = A.indices.data();
    SfCsrvData D;
    sf_csrv_data(a, A.values.data(), std::min(max_fmt, (int)FMT_PK), D);
    out.fmt = D.fmt;
    out.bytes_per_pass = D.bytes_per_pass;
    out.stream = D.bytes_per_pass > STREAM_BYTES;
    CTL_TRY(upload_vec(h, &out.csr_ptr, A.indptr));
    CTL_TRY(upload_vec(h, &out.csr_cols, A.indices));
    CTL_TRY(upload_vec(h, &out.csr_rbase, D.rbase));
    CTL_TRY(upload_vec(h, &out.csr_dcol, D.dcol));
    if (D.fmt == FMT_PK) {
        CTL_TRY(upload_vec(h, &out.vcode, D.vcode));
        CTL_TRY(upload_vec(h, &out.vdict, D.vdict));
    } else {
        CTL_TRY(upload_vec(h, &out.csr_vals, A.values));
    }
    return CTL_OK;
}

namespace {

constexpr int ST = 128;      // threads per CTA of the kernels in this file (the one-row-per-thread kernels of a large
                             // level run 256: BIG_BLOCK_ROWS)
constexpr int SC = 8;        // SELL entries fetched per thread before the first dependent gather

// ---- a gathered vector on the device: owned entries, and the ghosts either plainly stored (completed earlier) or
// in the slot of the exchange that delivers them (halo.cuh)
struct DVec {
    const double *x, *ghost;
    const ulonglong2 *ll;
    int n_own;
    unsigned idx1;
};

// seq_hi: the epoch bits of the running sequence numbers (halo_epoch_bits), read once per thread
__device__ __forceinline__ double dvec_get(const DVec &v, int c, unsigned seq_hi, const HaloCtx &ctx)
{
    if (c < v.n_own) return v.x[c];      // (a plain load: see the note on read-only loads below)
    if (v.ll) return halo_ll_read(v.ll + (c - v.n_own), seq_hi | v.idx1, ctx);
    return __ldcg(v.ghost + (c - v.n_own));
}

// ---- several components per row (block-scalar sweeps, one GPU: no ghosts, no push).  The matrix is the scalar S
// of I_NC (x) S; a row of S produces NC results and every gather loads the NC interleaved values of a node
// (dof = NC node + comp), one 16-byte load for NC = 2.  NC = 1 is the plain scalar path (vec_t<1> = double).
template <int NC>
struct VN {
    double c[NC];
};
template <int NC>
using vec_t = typename std::conditional<NC == 1, double, VN<NC>>::type;

template <int NC>
__device__ __forceinline__ VN<NC> operator+(VN<NC> a, const VN<NC> &b)
{
#pragma unroll
    for (int k = 0; k < NC; ++k) a.c[k] = a.c[k] + b.c[k];
    return a;
}
template <int NC>
__device__ __forceinline__ VN<NC> operator-(VN<NC> a, const VN<NC> &b)
{
#pragma unroll
    for (int k = 0; k < NC; ++k) a.c[k] = a.c[k] - b.c[k];
    return a;
}
template <int NC>
__device__ __forceinline__ VN<NC> operator*(double s, VN<NC> a)
{
#pragma unroll
    for (int k = 0; k < NC; ++k) a.c[k] = s * a.c[k];
    return a;
}
__device__ __forceinline__ double vfma(double a, double x, double acc) { return fma(a, x, acc); }
template <int NC>
__device__ __forceinline__ VN<NC> vfma(double a, const VN<NC> &x, VN<NC> acc)
{
#pragma unroll
    for (int k = 0; k < NC; ++k) acc.c[k] = fma(a, x.c[k], acc.c[k]);
    return acc;
}
__device__ __forceinline__ double vshfl_add(double v, int o, int w) { return v + __shfl_xor_sync(0xffffffffu, v, o, w); }
template <int NC>
__device__ __forceinline__ VN<NC> vshfl_add(VN<NC> v, int o, int w)
{
#pragma unroll
    for (int k = 0; k < NC; ++k) v.c[k] = v.c[k] + __shfl_xor_sync(0xffffffffu, v.c[k], o, w);
    return v;
}
// the NC values of node c (a plain load: vectors are written by the chain).  16-byte aligned for NC = 2: the vectors
// start 16-byte aligned and have an even number of entries on one GPU.
template <int NC>
__device__ __forceinline__ vec_t<NC> ld_node(const double *x, int c)
{
    if constexpr (NC == 1) {
        return x[c];
    } else if constexpr (NC == 2) {
        const double2 v = *reinterpret_cast<const double2 *>(x + 2 * c);
        VN<2> r;
        r.c[0] = v.x;
        r.c[1] = v.y;
        return r;
    } else {
        VN<NC> r;
#pragma unroll
        for (int k = 0; k < NC; ++k) r.c[k] = x[NC * c + k];
        return r;
    }
}
__device__ __forceinline__ void st_node(double *out, int row, double v) { out[row] = v; }
template <int NC>
__device__ __forceinline__ void st_node(double *out, int row, const VN<NC> &v)
{
    if constexpr (NC == 2) {
        *reinterpret_cast<double2 *>(out + 2 * row) = make_double2(v.c[0], v.c[1]);
    } else {
#pragma unroll
        for (int k = 0; k < NC; ++k) out[NC * row + k] = v.c[k];
    }
}
// a gathered vector of NC components (NC > 1: one GPU, so no ghost entries)
template <int NC>
__device__ __forceinline__ vec_t<NC> gat(const DVec &v, int c, unsigned seq_hi, const HaloCtx &ctx)
{
    if constexpr (NC == 1) return dvec_get(v, c, seq_hi, ctx);
    else return ld_node<NC>(v.x, c);
}

// READ-ONLY LOADS.  Vectors that a kernel of the chain writes (iterates, right-hand sides, residuals) are read with
// PLAIN loads in this file, never with __ldg / through a const __restrict__ parameter: ptxas orders a plain ld.global
// against griddepcontrol.wait but moves a non-coherent one (LDG.CONSTANT) freely -- with the wait no longer the first
// instruction of the kernel it hoisted the gathers of the iterate above it (as soon as their column indices had
// arrived), i.e. read the predecessor's output before the predecessor had finished: wrong sweeps on the GPU, caught
// by the parity tests.  Constant data (matrices, dinv) keeps __ldg: hoisting those is the point.
//
// Every row-dot helper below follows one schedule (pdl.cuh, pdl_trigger / pdl_wait): the loads of the MATRIX
// stream of the first chunk are issued first (constant data), then pdl_wait(), then `pre()` -- the caller's loads of
// the vector entries of its own row -- and only then the dependent gathers.  What a thread of the chain waits for
// after its predecessor has finished is ONE round trip (gathers and own-row loads together), not three.
//
// FMT_STENCIL: a slice whose 32 rows share one stencil reads (delta_k, value_k) through warp-uniform loads and
// gathers x[row + delta_k] (coalesced); the other slices take the per-entry DICT16 path.
// g: gather of a column that may be a ghost; g_own: gather of a column known to be owned (no ghost test)
template <typename G, typename G0, typename PRE>
__device__ __forceinline__ auto sell_row_dot_stencil(const MatView &A, int row, G g, G0 g_own, PRE pre)
{
    const int s = row >> 5, lane = row & 31;
    const int4 s0 = pre_ld(A.sp4 + s);
    // the most frequent stencil travels with the kernel parameters.  Whether its gathers would all stay inside the
    // owned columns is known from the row number alone, so they are issued SPECULATIVELY, together with the slice
    // descriptor: the common slice (99.6 % at C2) costs no dependent round trip for its descriptor, the others
    // throw eight loads away.
    const int first = s << 5;
    const bool spec = A.ps_w > 0 && first + A.ps_dmin >= 0 && first + 31 + A.ps_dmax < A.n_own;
    pdl_wait();
    pre();
    using R = decltype(g(0));
    R acc{};
    if (spec) {
        R xv[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) xv[j] = (j < A.ps_w) ? g_own(row + A.ps_delta[j]) : R{};
        if (s0.z == A.ps_off) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (j < A.ps_w) acc = vfma(A.ps_v[j], xv[j], acc);
            if (A.ps_w > 8) {      // second half (a P1 tetrahedron stencil has 15 entries)
#pragma unroll
                for (int j = 0; j < 8; ++j) xv[j] = (8 + j < A.ps_w) ? g_own(row + A.ps_delta[8 + j]) : R{};
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (8 + j < A.ps_w) acc = vfma(A.ps_v[8 + j], xv[j], acc);
            }
            return acc;
        }
    } else if (s0.z == A.ps_off) {
        // the same stencil next to a partition boundary: ghost-aware gathers, in two halves of 8
#pragma unroll
        for (int h0 = 0; h0 < SF_PS; h0 += 8) {
            if (h0 < A.ps_w) {
                R xv[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) xv[j] = (h0 + j < A.ps_w) ? g(row + A.ps_delta[h0 + j]) : R{};
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (h0 + j < A.ps_w) acc = vfma(A.ps_v[h0 + j], xv[j], acc);
            }
        }
        return acc;
    }
    if (s0.z >= 0) {
        // offsets first (warp-uniform 4-byte loads), then all gathers of the chunk, the values only when they are
        // multiplied: few live registers, all gathers in flight together
        const DictEnt *st = A.stab + s0.z;
        for (int k0 = 0; k0 < s0.y; k0 += SC) {
            int d[SC];
#pragma unroll
            for (int j = 0; j < SC; ++j)
                if (k0 + j < s0.y) d[j] = __ldg(&st[k0 + j].delta);
            R xv[SC];
#pragma unroll
            for (int j = 0; j < SC; ++j) xv[j] = (k0 + j < s0.y) ? g(row + d[j]) : R{};
#pragma unroll
            for (int j = 0; j < SC; ++j)
                if (k0 + j < s0.y) acc = vfma(__ldg(&st[k0 + j].v), xv[j], acc);
        }
        return acc;
    }
    // the few slices at mesh / partition boundaries: per-entry codes, one entry at a time
    const int end = s0.x + 32 * s0.y;
    const uint16_t *code = reinterpret_cast<const uint16_t *>(A.code);
#pragma unroll 1
    for (int p = s0.x + lane; p < end; p += 32) {
        const DictEnt e = sf_dict(A.dict, __ldg(code + p));
        acc = vfma(e.v, g(row + e.delta), acc);
    }
    return acc;
}

// One row of a SELL-32 slice.  The slice width is uniform across the warp, so the loop is divergence free;
// entries are fetched in chunks of SC with all stream loads issued before the dependent gathers
// (memory-level parallelism instead of a serial load -> gather -> fma chain per entry).
template <int FMT, bool STREAM, typename G, typename G0, typename PRE>
__device__ __forceinline__ auto sell_row_dot(const MatView &A, int row, G g, G0 g_own, PRE pre)
{
    if (FMT == FMT_STENCIL) return sell_row_dot_stencil(A, row, g, g_own, pre);
    const int s = row >> 5, lane = row & 31;
    const int2 s0 = pre_ld(A.sp + s);
    const int end = pre_ld(reinterpret_cast<const int *>(A.sp + s + 1));
    using R = decltype(g(0));
    R acc{};
    // chunk 0: its stream loads are issued before the wait for the predecessor grid
    auto chunk = [&](int p0, auto first) {
        constexpr bool PRE = decltype(first)::value;
        SfRaw raw[SC];
#pragma unroll
        for (int j = 0; j < SC; ++j) {
            const int p = p0 + 32 * j;
            if (p < end) raw[j] = sf_load<FMT, STREAM, PRE>(A, p);
        }
        if (PRE) {
            pdl_wait();
            pre();
        }
        int c[SC];
        double v[SC];
#pragma unroll
        for (int j = 0; j < SC; ++j) {
            const int p = p0 + 32 * j;
            if (p < end) {
                sf_decode<FMT>(A, raw[j], p, row, s0.y, c[j], v[j]);
            } else {
                c[j] = 0;
                v[j] = 0.0;
            }
        }
        R xv[SC];
#pragma unroll
        for (int j = 0; j < SC; ++j) xv[j] = g(c[j]);
#pragma unroll
        for (int j = 0; j < SC; ++j) acc = vfma(v[j], xv[j], acc);
    };
    int p0 = s0.x + lane;
    chunk(p0, std::true_type());      // (a slice without entries loads nothing and only waits)
    for (p0 += 32 * SC; p0 < end; p0 += 32 * SC) chunk(p0, std::false_type());
    return acc;
}

// format known only at run time (kernels that are not hot enough for one instantiation per format)
template <typename G>
__device__ __forceinline__ auto sell_row_dot_rt(const MatView &A, int row, G g)
{
    auto none = [] {};
    switch (A.fmt) {
    case FMT_F64: return sell_row_dot<FMT_F64, false>(A, row, g, g, none);
    case FMT_D16: return sell_row_dot<FMT_D16, false>(A, row, g, g, none);
    case FMT_PK: return sell_row_dot<FMT_PK, false>(A, row, g, g, none);
    case FMT_DICT16: return sell_row_dot<FMT_DICT16, false>(A, row, g, g, none);
    case FMT_STENCIL: return sell_row_dot_stencil(A, row, g, g, none);
    default: return sell_row_dot<FMT_DICT8, false>(A, row, g, g, none);
    }
}

// T lanes of a warp share one CSR row; the result is valid on every lane of the group.  A lane fetches its
// entries in chunks of CU with the stream loads issued before the dependent gathers (the rows of the restrictions
// and of R A are long: a serial load -> gather chain per entry is what these latency-bound kernels cannot afford).
constexpr int CU = 4;
template <int T, int FMT, bool STREAM, typename G, typename PRE>
__device__ __forceinline__ auto csrv_row_dot_f(const MatView &A, int row, int sub, G g, PRE pre)
{
    const int beg = pre_ld(A.ptr + row), end = pre_ld(A.ptr + row + 1);
    const int base = (FMT == FMT_F64) ? 0 : pre_ld(A.rbase + row);
    using R = decltype(g(0));
    R acc{};
    auto chunk = [&](int p0, auto first) {
        constexpr bool PRE = decltype(first)::value;
        SfRaw raw[CU];
#pragma unroll
        for (int j = 0; j < CU; ++j)
            if (p0 + j * T < end) raw[j] = sf_load<FMT, STREAM, PRE>(A, p0 + j * T);
        if (PRE) {
            pdl_wait();
            pre();
        }
        int c[CU];
        double v[CU];
#pragma unroll
        for (int j = 0; j < CU; ++j) {
            if (p0 + j * T < end) {
                sf_decode<FMT>(A, raw[j], p0 + j * T, row, base, c[j], v[j]);
            } else {
                c[j] = 0;
                v[j] = 0.0;
            }
        }
        R xv[CU];
#pragma unroll
        for (int j = 0; j < CU; ++j) xv[j] = g(c[j]);
#pragma unroll
        for (int j = 0; j < CU; ++j) acc = vfma(v[j], xv[j], acc);
    };
    int p0 = beg + sub;
    chunk(p0, std::true_type());      // (a lane without entries of its own loads nothing and only waits)
    for (p0 += CU * T; p0 < end; p0 += CU * T) chunk(p0, std::false_type());
#pragma unroll
    for (int o = T / 2; o > 0; o >>= 1) acc = vshfl_add(acc, o, T);
    return acc;
}

template <int T, bool STREAM, typename G, typename PRE>
__device__ __forceinline__ auto csrv_row_dot(const MatView &A, int row, int sub, G g, PRE pre)
{
    if (A.fmt == FMT_F64) return csrv_row_dot_f<T, FMT_F64, STREAM>(A, row, sub, g, pre);
    if (A.fmt == FMT_D16) return csrv_row_dot_f<T, FMT_D16, STREAM>(A, row, sub, g, pre);
    return csrv_row_dot_f<T, FMT_PK, STREAM>(A, row, sub, g, pre);
}

// Row assignment shared by every kernel: the push CTAs (halo.cuh) come first and compute the listed boundary
// rows, one chunk of <= 32 rows per warp, storing them locally and into the ghost slots of the ranks that gather
// them; the regular CTAs compute ST / T consecutive rows each.  f(row) is evaluated by all T lanes of a row's
// group and returns the value to store in out[row] (NC components: the NC values of out at row's node; such rows are
// never pushed).
template <int T, int BS = ST, typename F>
__device__ __forceinline__ void run_rows(int n_rows, const HaloPush &push, unsigned seq_hi, double *out, F f)
{
    using R = decltype(f(0));
    constexpr bool SCALAR = std::is_same<R, double>::value;
    constexpr int RPC = BS / T;
    const int n_pc = SCALAR ? (push.n_chunks + BS / 32 - 1) / (BS / 32) : 0;
    if constexpr (SCALAR) {
    const int lane = threadIdx.x & 31;
    if ((int)blockIdx.x < n_pc) {
        const int ci = blockIdx.x * (BS / 32) + (threadIdx.x >> 5);
        if (ci >= push.n_chunks) {
            pdl_wait();      // no thread leaves before the predecessor is complete: grids finish in launch order
            return;
        }
        const PushChunk ch = push.chunks[ci];
        const unsigned seq = seq_hi | push.idx1;
#pragma unroll 1
        for (int pass = 0; pass < T; ++pass) {
            const int idx = pass * (32 / T) + lane / T;
            const bool live = idx < ch.count;
            const int row = push.rows[ch.start + (live ? idx : 0)];
            const double v = f(row);
            if (live && (lane % T) == 0) {
                out[row] = v;
                for (int d = 0; d < ch.n_dst; ++d) {
                    const PushDst t = push.dsts[ch.dst_begin + d];
                    halo_ll_store(t.base + (long long)push.slot * t.stride + t.pos[idx], v, seq);
                }
            }
        }
        return;
    }
    if (push.all_rows) {
        pdl_wait();
        return;
    }
    }
    const int r0 = ((int)blockIdx.x - n_pc) * RPC;
    const int row = r0 + (int)threadIdx.x / T;
    if (T == 1) {
        if (row < n_rows) st_node(out, row, f(row));
        else pdl_wait();      // no thread leaves before the predecessor is complete: grids finish in launch order
    } else {
        const bool live = row < n_rows;
        const R v = f(live ? row : n_rows - 1);
        if (live && (threadIdx.x % T) == 0) st_node(out, row, v);
    }
}

// kernel-side modes: y = A x | b - A x | b + sign A x (ADD / SUB arrive as b = y); bi = b[row], loaded by the caller
__device__ __forceinline__ double apply_mode(int mode, double ax, double bi)
{
    if (mode == SELL_ASSIGN) return ax;
    if (mode == SELL_RESIDUAL) return bi - ax;
    return bi + ax;      // SELL_BPLUS
}
template <int NC>
__device__ __forceinline__ VN<NC> apply_mode(int mode, const VN<NC> &ax, const VN<NC> &bi)
{
    if (mode == SELL_ASSIGN) return ax;
    if (mode == SELL_RESIDUAL) return bi - ax;
    return bi + ax;
}

// Start of every kernel of this file: let the successor be scheduled and read the epoch bits of the exchange's
// sequence numbers.  The wait for the predecessor happens inside the row-dot helpers, after the loads of the matrix
// stream.  (The epoch word is bumped once per replay behind a complete kernel boundary, halo.cu::halo_epoch_begin,
// so it may be read before the wait.)
__device__ __forceinline__ unsigned kernel_prologue(const HaloCtx &ctx)
{
    pdl_trigger();
    if (!ctx.epoch) return 0u;
    if (ctx.early_wait) pdl_wait();
    return halo_epoch_bits(ctx);
}

// ---------------------------------------------------------------- SELL kernels
// GH: the gathered vector has ghost entries (several GPUs); without them the gather is a plain read-only load
template <int FMT, bool STREAM, bool GH, int BS, int NC>
__global__ void __launch_bounds__(BS) sell_spmv_kernel(const MatView A, const DVec x, const HaloCtx ctx, const double *b,
                                                      double *y, int mode, double sign, const HaloPush push)
{
    const unsigned hi = kernel_prologue(ctx);
    run_rows<1, BS>(A.n_rows, push, hi, y, [&](int row) {
        vec_t<NC> bi{};
        const vec_t<NC> ax = sign * sell_row_dot<FMT, STREAM>(
                                     A, row, [&](int c) { if constexpr (GH) return dvec_get(x, c, hi, ctx); else return ld_node<NC>(x.x, c); },
                                     [&](int c) { return ld_node<NC>(x.x, c); },
                                     [&] { if (mode != SELL_ASSIGN) bi = ld_node<NC>(b, row); });
        return apply_mode(mode, ax, bi);
    });
}

// one Chebyshev step; the loads of the row's own entries (b, p_cur, p_prev) travel with the gathers
#define CHEB_ROW_UPDATE(DOT)                                                                              \
    const double di = pre_ld(dinv + row);      /* constant: before the wait; one per node */               \
    vec_t<NC> bi{}, pc{}, pp{};                                                                           \
    auto pre = [&] {                                                                                      \
        bi = ld_node<NC>(b, row);                                                                         \
        pc = ld_node<NC>(p_cur.x, row);                                                                   \
        if (prev_scale == 0.0 && a != 0.0) pp = ld_node<NC>(p_prev, row);                                 \
    };                                                                                                    \
    const vec_t<NC> ax = DOT;                                                                             \
    vec_t<NC> r = bq * pc + c * di * (bi - ax);                                                           \
    if (prev_scale != 0.0) r = vfma(a, prev_scale * di * bi, r);                                          \
    else if (a != 0.0) r = vfma(a, pp, r);                                                                \
    return r

template <int FMT, bool STREAM, bool GH, int BS, int NC>
__global__ void __launch_bounds__(BS) sell_cheb_kernel(const MatView A, const double *__restrict__ dinv,
                                                      const double *b, const double *p_prev, const DVec p_cur,
                                                      const HaloCtx ctx, double *out, double a, double bq, double c,
                                                      double prev_scale, const HaloPush push)
{
    const unsigned hi = kernel_prologue(ctx);
    run_rows<1, BS>(A.n_rows, push, hi, out, [&](int row) {
        CHEB_ROW_UPDATE((sell_row_dot<FMT, STREAM>(
            A, row, [&](int cc) { if constexpr (GH) return dvec_get(p_cur, cc, hi, ctx); else return ld_node<NC>(p_cur.x, cc); },
            [&](int cc) { return ld_node<NC>(p_cur.x, cc); }, pre)));
    });
}

template <int FMT, bool STREAM, bool GH, int BS, int NC>
__global__ void __launch_bounds__(BS) sell_first2_kernel(const MatView A, const DVec dinv, const DVec b, const HaloCtx ctx,
                                                        double *out, double s, double wgt, const HaloPush push)
{
    const unsigned hi = kernel_prologue(ctx);
    run_rows<1, BS>(A.n_rows, push, hi, out, [&](int row) {
        const double di = pre_ld(dinv.x + row);
        vec_t<NC> bi{};
        const vec_t<NC> ax = sell_row_dot<FMT, STREAM>(
            A, row,
            [&](int c) {
                if constexpr (GH) return s * dvec_get(dinv, c, hi, ctx) * dvec_get(b, c, hi, ctx);
                else return s * __ldg(dinv.x + c) * ld_node<NC>(b.x, c);
            },
            [&](int c) { return s * __ldg(dinv.x + c) * ld_node<NC>(b.x, c); }, [&] { bi = ld_node<NC>(b.x, row); });
        const vec_t<NC> p1 = s * di * bi;
        return wgt * p1 + (wgt * s) * di * (bi - ax);
    });
}

template <int NC>
__global__ void __launch_bounds__(ST) sell_spmv2_kernel(const MatView A1, const MatView A2, const DVec x1, const DVec x2,
                                                       const DVec x3, double *y, double alpha, double beta,
                                                       const HaloCtx ctx, const HaloPush push)
{
    const unsigned hi = kernel_prologue(ctx);
    run_rows<1>(A1.n_rows, push, hi, y, [&](int row) {
        vec_t<NC> acc1;
        if (x2.x) acc1 = sell_row_dot_rt(A1, row, [&](int c) { return gat<NC>(x1, c, hi, ctx) + gat<NC>(x2, c, hi, ctx); });
        else acc1 = sell_row_dot_rt(A1, row, [&](int c) { return gat<NC>(x1, c, hi, ctx); });
        vec_t<NC> acc2{};
        if (x3.x) acc2 = sell_row_dot_rt(A2, row, [&](int c) { return gat<NC>(x3, c, hi, ctx); });
        return alpha * acc1 + beta * acc2;
    });
}

template <int NC>
__global__ void __launch_bounds__(ST) dinv_scale_kernel(const double *__restrict__ dinv, const double *b,
                                                       double *out, double c, int n, const HaloCtx ctx,
                                                       const HaloPush push)
{
    const unsigned hi = kernel_prologue(ctx);
    run_rows<1>(n, push, hi, out, [&](int row) {
        const double di = pre_ld(dinv + row);
        pdl_wait();
        return c * di * ld_node<NC>(b, row);
    });
}

// Small dense matrix (the coarsest level: 2205 rows at C2, 39 MB, L2-resident), rows padded to `lda` (even: every
// row starts 16-byte aligned).  One CTA per GR rows, so that b is read once per GR rows; a thread keeps GU x GR
// independent 16-byte loads of the matrix in flight, and the first batch of them is issued BEFORE the wait for the
// predecessor (the matrix is constant).  Round 2: 15 us -> see profiles/r02_*: the first version walked odd-sized
// rows with 8-byte loads, four per thread and iteration.
constexpr int GR = 4;
constexpr int GU = 2;
template <int NC>
__global__ void __launch_bounds__(ST) dense_gemv_kernel(const double *__restrict__ A, const double *b,
                                                       double *y, int n, int lda)
{
    using R = vec_t<NC>;
    pdl_trigger();
    __shared__ R part[GR][ST / 32];
    const int r0 = blockIdx.x * GR;
    R acc[GR];
#pragma unroll
    for (int q = 0; q < GR; ++q) acc[q] = R{};
    const int n2 = n >> 1;      // complete pairs; an odd last column is handled below (the padding column is zero)
    const bool b_aligned = (reinterpret_cast<uintptr_t>(b) & 15) == 0;
    const double2 *rowp[GR];
#pragma unroll
    for (int q = 0; q < GR; ++q) rowp[q] = reinterpret_cast<const double2 *>(A + (size_t)min(r0 + q, n - 1) * lda);
    bool waited = false;
    for (int j0 = threadIdx.x; j0 < n2; j0 += GU * ST) {
        double2 av[GU][GR];
#pragma unroll
        for (int u = 0; u < GU; ++u) {
            const int j = j0 + u * ST;
#pragma unroll
            for (int q = 0; q < GR; ++q) av[u][q] = (j < n2) ? pre_ld(rowp[q] + j) : make_double2(0.0, 0.0);
        }
        if (!waited) {
            pdl_wait();
            waited = true;
        }
        R bx[GU], by[GU];      // b at the columns 2j and 2j + 1
#pragma unroll
        for (int u = 0; u < GU; ++u) {
            const int j = j0 + u * ST;
            if (j >= n2) {
                bx[u] = R{};
                by[u] = R{};
            } else if constexpr (NC == 1) {
                const double2 t = b_aligned ? reinterpret_cast<const double2 *>(b)[j] : make_double2(b[2 * j], b[2 * j + 1]);
                bx[u] = t.x;
                by[u] = t.y;
            } else {
                bx[u] = ld_node<NC>(b, 2 * j);
                by[u] = ld_node<NC>(b, 2 * j + 1);
            }
        }
#pragma unroll
        for (int u = 0; u < GU; ++u)
#pragma unroll
            for (int q = 0; q < GR; ++q) acc[q] = vfma(av[u][q].y, by[u], vfma(av[u][q].x, bx[u], acc[q]));
    }
    if (!waited) pdl_wait();
    if ((n & 1) && threadIdx.x == 0) {
        const R bl = ld_node<NC>(b, n - 1);
#pragma unroll
        for (int q = 0; q < GR; ++q) acc[q] = vfma(__ldg(A + (size_t)min(r0 + q, n - 1) * lda + n - 1), bl, acc[q]);
    }
#pragma unroll
    for (int q = 0; q < GR; ++q) {
        R s = acc[q];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s = vshfl_add(s, o, 32);
        if ((threadIdx.x & 31) == 0) part[q][threadIdx.x >> 5] = s;
    }
    __syncthreads();
    if (threadIdx.x < GR && r0 + threadIdx.x < n)
    {
        R s{};
#pragma unroll
        for (int w = 0; w < ST / 32; w += 4)      // fixed order: pairs first
            s = s + ((part[threadIdx.x][w] + part[threadIdx.x][w + 1]) + (part[threadIdx.x][w + 2] + part[threadIdx.x][w + 3]));
        st_node(y, r0 + threadIdx.x, s);
    }
}

// ---------------------------------------------------------------- CSR-vector kernels
template <int T, bool STREAM, int NC>
__global__ void __launch_bounds__(ST) csrv_spmv_kernel(const MatView A, const DVec x, const HaloCtx ctx, const double *b,
                                                      double *y, int mode, double sign, const HaloPush push)
{
    const unsigned hi = kernel_prologue(ctx);
    const int sub = threadIdx.x % T;
    run_rows<T>(A.n_rows, push, hi, y, [&](int row) {
        vec_t<NC> bi{};
        const vec_t<NC> ax = sign * csrv_row_dot<T, STREAM>(A, row, sub, [&](int c) { return gat<NC>(x, c, hi, ctx); },
                                                            [&] { if (mode != SELL_ASSIGN) bi = ld_node<NC>(b, row); });
        return apply_mode(mode, ax, bi);
    });
}

template <int T, int NC>
__global__ void __launch_bounds__(ST) csrv_cheb_kernel(const MatView A, const double *__restrict__ dinv,
                                                      const double *b, const double *p_prev, const DVec p_cur,
                                                      const HaloCtx ctx, double *out, double a, double bq, double c,
                                                      double prev_scale, const HaloPush push)
{
    const unsigned hi = kernel_prologue(ctx);
    const int sub = threadIdx.x % T;
    run_rows<T>(A.n_rows, push, hi, out, [&](int row) {
        CHEB_ROW_UPDATE((csrv_row_dot<T, false>(A, row, sub, [&](int cc) { return gat<NC>(p_cur, cc, hi, ctx); }, pre)));
    });
}

template <int T, int NC>
__global__ void __launch_bounds__(ST) csrv_first2_kernel(const MatView A, const DVec dinv, const DVec b, const HaloCtx ctx,
                                                        double *out, double s, double wgt, const HaloPush push)
{
    const unsigned hi = kernel_prologue(ctx);
    const int sub = threadIdx.x % T;
    run_rows<T>(A.n_rows, push, hi, out, [&](int row) {
        const double di = pre_ld(dinv.x + row);
        vec_t<NC> bi{};
        const vec_t<NC> ax = csrv_row_dot<T, false>(A, row, sub, [&](int c) { return s * dvec_get(dinv, c, hi, ctx) * gat<NC>(b, c, hi, ctx); },
                                                    [&] { bi = ld_node<NC>(b.x, row); });
        const vec_t<NC> p1 = s * di * bi;
        return wgt * p1 + (wgt * s) * di * (bi - ax);
    });
}

DVec dvec(const GVec &g, const MatView &A)
{
    DVec d;
    d.x = g.x;
    d.ghost = g.ghost;
    d.ll = g.ll;
    d.n_own = A.n_own;
    d.idx1 = g.idx1;
    return d;
}

bool has_ghosts(const GVec &g) { return g.ghost != nullptr || g.ll != nullptr; }

// components run on one GPU only: no ghost entries, no pushed rows
int check_nc(ctl_handle_s *h, const SellMat &A, bool ghosts, const HaloPush &push, const char *what)
{
    CTL_CHECK(A.nc == 1 || (!ghosts && push.n_chunks == 0 && !push.all_rows), CTL_ERR_STATE,
              std::string(what) + ": matrices with several components run on one GPU only");
    return CTL_OK;
}

// push CTAs first; a replicating exchange pushes every row, so the regular CTAs are not launched at all
int grid_for(int n_rows, int T, const HaloPush &push, int bs = ST)
{
    if (push.all_rows) return halo_push_ctas(push, bs);
    return ceil_div((int64_t)n_rows * T, bs) + halo_push_ctas(push, bs);
}

// CTAs of 256 threads for the one-row-per-thread kernels of a LARGE level on one GPU: the 1 M-row kernels of C2 are
// bound by launch ramp and tail of their 8209 small CTAs (43 % of the warp slots active, ncu), and half as many CTAs
// of twice the size take 11-15 % off them (smoother step 11.95 -> 10.63 us, residual 11.76 -> 10.02 us, measured with
// an all-256 build: profiles/r02_inner_solve_variants.txt); the small levels lose with fewer, larger CTAs and keep 128,
// and so do long rows (the 15-point stencil of C3: its level-0 smoother went from 53 to 58 us with 256-thread CTAs).
constexpr int BIG_BLOCK_ROWS = 400000;

// ---- launch dispatch: the run-time choices become the compile-time parameters of the kernel templates
template <int V>
using int_c = std::integral_constant<int, V>;
template <bool V>
using bool_c = std::integral_constant<bool, V>;

// f(NC) for the component counts of the block-scalar sweeps
template <typename F>
void with_nc(int nc, F f)
{
    if (nc == 2) f(int_c<2>());
    else if (nc == 3) f(int_c<3>());
    else f(int_c<1>());
}

// f(T) for the lanes per row of a CSR-vector matrix
template <typename F>
void with_lanes(int lanes, F f)
{
    if (lanes == 4) f(int_c<4>());
    else if (lanes == 8) f(int_c<8>());
    else f(int_c<16>());
}

// A SELL kernel of A: f(grid, FMT, STREAM, GH, BS, NC), the last five compile-time.  Only the combinations that occur
// are instantiated: evict-first streaming only in the formats that read a plain value array (F64, D16, PK); ghosts
// (GH: a gathered vector has ghost entries) only with one component in CTAs of ST threads; CTAs of 256 threads only
// on one GPU without pushed rows.  Returns false and launches nothing when the grid is empty.
template <typename F>
bool sell_dispatch(const SellMat &A, bool ghosts, const HaloPush &push, F f)
{
    const bool big = !ghosts && push.n_chunks == 0 && A.pat->n_rows >= BIG_BLOCK_ROWS && A.pat->nnz <= 10ll * A.pat->n_rows;
    const int grid = grid_for(A.pat->n_rows, 1, push, big ? 256 : ST);
    if (grid == 0) return false;
    auto launch = [&](auto fmt, auto stream) {
        with_nc(A.nc, [&](auto nc) {
            if constexpr (decltype(nc)::value == 1) {
                if (ghosts) {
                    f(grid, fmt, stream, bool_c<true>(), int_c<ST>(), nc);
                    return;
                }
            }
            if (big) f(grid, fmt, stream, bool_c<false>(), int_c<256>(), nc);
            else f(grid, fmt, stream, bool_c<false>(), int_c<ST>(), nc);
        });
    };
    auto with_stream = [&](auto fmt) {
        constexpr int FMT = decltype(fmt)::value;
        if constexpr (FMT == FMT_F64 || FMT == FMT_D16 || FMT == FMT_PK) {
            if (A.stream) {
                launch(fmt, bool_c<true>());
                return;
            }
        }
        launch(fmt, bool_c<false>());
    };
    switch (A.fmt) {
    case FMT_F64: with_stream(int_c<FMT_F64>()); break;
    case FMT_D16: with_stream(int_c<FMT_D16>()); break;
    case FMT_PK: with_stream(int_c<FMT_PK>()); break;
    case FMT_DICT16: with_stream(int_c<FMT_DICT16>()); break;
    case FMT_STENCIL: with_stream(int_c<FMT_STENCIL>()); break;
    default: with_stream(int_c<FMT_DICT8>()); break;
    }
    return true;
}

// A CSR-vector kernel of A (CTAs of ST threads): f(grid, T, NC), the last two compile-time.  Returns false and launches
// nothing when the grid is empty.
template <typename F>
bool csrv_dispatch(const SellMat &A, const HaloPush &push, F f)
{
    const int grid = grid_for(A.pat->n_rows, A.lanes, push);
    if (grid == 0) return false;
    with_lanes(A.lanes, [&](auto T) { with_nc(A.nc, [&](auto nc) { f(grid, T, nc); }); });
    return true;
}

}  // namespace

int sell_spmv(ctl_handle_s *h, const SellMat &A, const GVec &x, double *y, const double *b, int mode, const HaloPush &push)
{
    // y (+)= / -= A x: expressed as y = b +/- A x with b = y; aliasing is not idempotent, so a pushing launch
    // (whose boundary rows are computed twice) must not use it
    double sign = 1.0;
    int kmode = mode;
    if (mode == SELL_ADD || mode == SELL_SUB) {
        b = y;
        kmode = SELL_BPLUS;
        sign = mode == SELL_SUB ? -1.0 : 1.0;
    }
    CTL_CHECK(kmode == SELL_ASSIGN || b != nullptr, CTL_ERR_ARG, "sell_spmv: this mode needs b");
    CTL_CHECK(push.n_chunks == 0 || b != y, CTL_ERR_STATE, "sell_spmv: an in-place product cannot push its boundary rows");
    CTL_TRY(check_nc(h, A, has_ghosts(x), push, "sell_spmv"));
    const MatView V = A.view();
    const DVec dx = dvec(x, V);
    const HaloCtx ctx = halo_ctx(h);
    bool launched;
    if (A.lanes) {
        launched = csrv_dispatch(A, push, [&](int grid, auto T, auto NC) {
            if (A.stream) pdl_launch(h, grid, ST, csrv_spmv_kernel<T, true, NC>, V, dx, ctx, b, y, kmode, sign, push);
            else pdl_launch(h, grid, ST, csrv_spmv_kernel<T, false, NC>, V, dx, ctx, b, y, kmode, sign, push);
        });
    } else {
        launched = sell_dispatch(A, has_ghosts(x), push, [&](int grid, auto F, auto S, auto G, auto B, auto NC) {
            pdl_launch(h, grid, B, sell_spmv_kernel<F, S, G, B, NC>, V, dx, ctx, b, y, kmode, sign, push);
        });
    }
    if (!launched) return CTL_OK;
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

int sell_cheb_step(ctl_handle_s *h, const SellMat &A, const double *dinv, const double *b, const double *p_prev,
                   const GVec &p_cur, double *out, double a, double bq, double c, double prev_scale, const HaloPush &push)
{
    CTL_CHECK(push.n_chunks == 0 || (out != p_prev && out != p_cur.x), CTL_ERR_STATE,
              "sell_cheb_step: a pushing step must not overwrite its inputs");
    CTL_TRY(check_nc(h, A, has_ghosts(p_cur), push, "sell_cheb_step"));
    const MatView V = A.view();
    const DVec dx = dvec(p_cur, V);
    const HaloCtx ctx = halo_ctx(h);
    bool launched;
    if (A.lanes) {
        launched = csrv_dispatch(A, push, [&](int grid, auto T, auto NC) {
            pdl_launch(h, grid, ST, csrv_cheb_kernel<T, NC>, V, dinv, b, p_prev, dx, ctx, out, a, bq, c, prev_scale, push);
        });
    } else {
        launched = sell_dispatch(A, has_ghosts(p_cur), push, [&](int grid, auto F, auto S, auto G, auto B, auto NC) {
            pdl_launch(h, grid, B, sell_cheb_kernel<F, S, G, B, NC>, V, dinv, b, p_prev, dx, ctx, out, a, bq, c, prev_scale,
                       push);
        });
    }
    if (!launched) return CTL_OK;
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

int sell_cheb_first2(ctl_handle_s *h, const SellMat &A, const GVec &dinv, const GVec &b, double *out, double s, double w,
                     const HaloPush &push)
{
    const bool ghosts = has_ghosts(b) || has_ghosts(dinv);
    CTL_TRY(check_nc(h, A, ghosts, push, "sell_cheb_first2"));
    const MatView V = A.view();
    const DVec dd = dvec(dinv, V), db = dvec(b, V);
    const HaloCtx ctx = halo_ctx(h);
    bool launched;
    if (A.lanes) {
        launched = csrv_dispatch(A, push, [&](int grid, auto T, auto NC) {
            pdl_launch(h, grid, ST, csrv_first2_kernel<T, NC>, V, dd, db, ctx, out, s, w, push);
        });
    } else {
        launched = sell_dispatch(A, ghosts, push, [&](int grid, auto F, auto S, auto G, auto B, auto NC) {
            pdl_launch(h, grid, B, sell_first2_kernel<F, S, G, B, NC>, V, dd, db, ctx, out, s, w, push);
        });
    }
    if (!launched) return CTL_OK;
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

int vec_dinv_scale(ctl_handle_s *h, const double *dinv, const double *b, double *out, double c, int n, const HaloPush &push,
                   int nc)
{
    CTL_CHECK(nc == 1 || (push.n_chunks == 0 && !push.all_rows), CTL_ERR_STATE,
              "vec_dinv_scale: vectors with several components run on one GPU only");
    const int grid = grid_for(n, 1, push);
    if (grid == 0) return CTL_OK;
    with_nc(nc, [&](auto NC) { pdl_launch(h, grid, ST, dinv_scale_kernel<NC>, dinv, b, out, c, n, halo_ctx(h), push); });
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

int dense_gemv(ctl_handle_s *h, const double *Ainv, const double *b, double *y, int n, int lda, int nc)
{
    CTL_CHECK(lda >= n && (lda & 1) == 0, CTL_ERR_ARG, "dense_gemv: the row stride must be even and >= n");
    if (n == 0) return CTL_OK;
    with_nc(nc, [&](auto NC) { pdl_launch(h, ceil_div(n, GR), ST, dense_gemv_kernel<NC>, Ainv, b, y, n, lda); });
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

int sell_spmv2(ctl_handle_s *h, const SellMat &A1, const SellMat &A2, const GVec &x1, const GVec &x2, const GVec &x3,
               double *y, double alpha, double beta, const HaloPush &push)
{
    CTL_CHECK(A1.lanes == 0 && A2.lanes == 0, CTL_ERR_STATE, "sell_spmv2: SELL matrices only");
    CTL_CHECK(A1.nc == A2.nc, CTL_ERR_STATE, "sell_spmv2: both matrices need the same number of components");
    CTL_TRY(check_nc(h, A1, has_ghosts(x1) || has_ghosts(x2) || has_ghosts(x3), push, "sell_spmv2"));
    const int grid = grid_for(A1.pat->n_rows, 1, push);
    if (grid == 0) return CTL_OK;
    const MatView V1 = A1.view(), V2 = A2.view();
    const DVec d1 = dvec(x1, V1), d2 = dvec(x2, V1), d3 = dvec(x3, V2);
    const HaloCtx ctx = halo_ctx(h);
    with_nc(A1.nc, [&](auto NC) {
        pdl_launch(h, grid, ST, sell_spmv2_kernel<NC>, V1, V2, d1, d2, d3, y, alpha, beta, ctx, push);
    });
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

int vec_copy_n(ctl_handle_s *h, double *dst, const double *src, int n)
{
    CTL_CUDA(cudaMemcpyAsync(dst, src, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    return CTL_OK;
}
