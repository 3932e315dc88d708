// C ABI: handle lifetime, matrix hand-over, row partition, operator apply entry points.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "vec_ops.cuh"

static thread_local std::string g_create_error;

void ctl_set_error(ctl_handle_s *h, const std::string &msg)
{
    if (h) h->err = msg;
    else g_create_error = msg;
}

// PETSc's ownership split (PetscSplitOwnership): the first n % world ranks get one extra row
static void split_ownership(int n, int world, int rank, int *begin, int *count)
{
    const int base = n / world, rem = n % world;
    *count = base + (rank < rem ? 1 : 0);
    *begin = rank * base + std::min(rank, rem);
}

template <typename T>
int ctl_upload(ctl_handle_s *h, T **dst, const T *src, size_t count)
{
    if (*dst) {
        cudaFree(*dst);
        *dst = nullptr;
    }
    if (count == 0) return CTL_OK;
    CTL_CUDA(cudaMalloc((void **)dst, count * sizeof(T)));
    CTL_CUDA(cudaMemcpyAsync(*dst, src, count * sizeof(T), cudaMemcpyHostToDevice, h->stream));
    CTL_CUDA(cudaStreamSynchronize(h->stream));
    return CTL_OK;
}
template int ctl_upload<int>(ctl_handle_s *, int **, const int *, size_t);
template int ctl_upload<double>(ctl_handle_s *, double **, const double *, size_t);
template int ctl_upload<uint8_t>(ctl_handle_s *, uint8_t **, const uint8_t *, size_t);

extern "C" {

const char *ctl_version(void) { return "ctl_b200 0.1 (sm_100a)"; }

const char *ctl_last_error(ctl_handle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int ctl_create(const ctl_config *cfg, ctl_handle *out)
{
    ctl_handle_s *h = nullptr;
    CTL_CHECK(cfg && out, CTL_ERR_ARG, "ctl_create: null argument");
    CTL_CHECK(cfg->n > 0, CTL_ERR_ARG, "ctl_create: n must be positive");
    CTL_CHECK(cfg->n_t >= 2, CTL_ERR_ARG, "ctl_create: n_t must be at least 2");
    CTL_CHECK(cfg->tau > 0 && cfg->beta > 0, CTL_ERR_ARG, "ctl_create: tau and beta must be positive");
    CTL_CHECK(cfg->world >= 1 && cfg->rank >= 0 && cfg->rank < cfg->world, CTL_ERR_ARG,
              "ctl_create: bad rank/world");
    const int N = cfg->CN ? cfg->n_t - 1 : cfg->n_t;
    CTL_CHECK(N <= 256, CTL_ERR_ARG, "ctl_create: more than 256 time blocks are not supported");
    {
        cudaError_t e = cudaSetDevice(cfg->device);
        if (e != cudaSuccess) {
            ctl_set_error(nullptr, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
            return CTL_ERR_CUDA;
        }
    }
    h = new ctl_handle_s();
    h->cfg = *cfg;
    if (h->cfg.epsilon <= 0) h->cfg.epsilon = 1e-3;     // control/control.py:2836
    h->N = N;
    int ld = 8;
    while (ld < N) ld *= 2;
    h->ld = ld;
    h->n = cfg->n;
    split_ownership(cfg->n, cfg->world, cfg->rank, &h->row_begin, &h->n_loc);
    h->pool.init(h, std::max<int64_t>(h->vec_len(), 1));
    if (cfg->stream) {
        h->stream = (cudaStream_t)cfg->stream;
    } else {
        cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) {
            ctl_set_error(nullptr, std::string("cudaStreamCreate: ") + cudaGetErrorString(e));
            delete h;
            return CTL_ERR_CUDA;
        }
        h->own_stream = true;
    }
    h->h_bcmask.assign(cfg->n, 0);
    *out = h;
    return CTL_OK;
}

int ctl_destroy(ctl_handle h)
{
    if (!h) return CTL_OK;
    cudaSetDevice(h->cfg.device);
    cudaStreamSynchronize(h->stream);
    ctl_pc_free(h);
    ctl_comm_free(h);
    ctl_lift_invalidate(h);
    cudaFree(h->d_indptr);
    cudaFree(h->d_indices);
    cudaFree(h->d_M);
    cudaFree(h->d_M_full);
    if (h->d_KT != h->d_K) cudaFree(h->d_KT);
    cudaFree(h->d_K);
    cudaFree(h->d_bcmask);
    cudaFree(h->d_bc_rows_all);
    cudaFree(h->d_halo);
    cudaFree(h->d_red);
    if (h->h_red) cudaFreeHost(h->h_red);
    if (h->own_stream) cudaStreamDestroy(h->stream);
    delete h;
    return CTL_OK;
}

int ctl_set_pattern(ctl_handle h, const int32_t *indptr, const int32_t *indices, int64_t nnz)
{
    CTL_CHECK(h && indptr && indices, CTL_ERR_ARG, "ctl_set_pattern: null argument");
    CTL_CHECK(indptr[0] == 0 && indptr[h->n] == nnz, CTL_ERR_ARG,
              "ctl_set_pattern: indptr does not match n / nnz");
    for (int r = 0; r < h->n; ++r) {
        CTL_CHECK(indptr[r + 1] >= indptr[r], CTL_ERR_ARG, "ctl_set_pattern: indptr not monotone");
        for (int k = indptr[r]; k < indptr[r + 1]; ++k) {
            CTL_CHECK(indices[k] >= 0 && indices[k] < h->n, CTL_ERR_ARG,
                      "ctl_set_pattern: column index out of range");
            CTL_CHECK(k == indptr[r] || indices[k] > indices[k - 1], CTL_ERR_ARG,
                      "ctl_set_pattern: column indices must be sorted and unique within a row");
        }
    }
    h->h_indptr.assign(indptr, indptr + h->n + 1);
    h->h_tperm.clear();
    h->h_indices.assign(indices, indices + nnz);
    h->h_M.clear();
    h->h_K.clear();
    h->h_KT.clear();
    h->loc = HostCSR();
    ctl_lift_invalidate(h);
    h->assembled = false;
    return CTL_OK;
}

int ctl_set_values(ctl_handle h, int which, int level, const double *values)
{
    CTL_CHECK(h && values, CTL_ERR_ARG, "ctl_set_values: null argument");
    CTL_CHECK(!h->h_indptr.empty(), CTL_ERR_STATE, "ctl_set_values: call ctl_set_pattern first");
    const size_t nnz = h->h_indices.size();
    CTL_CHECK(level >= -1 && level < h->cfg.n_t, CTL_ERR_ARG, "ctl_set_values: bad level");
    if (which == CTL_MAT_M) {
        CTL_CHECK(level == -1, CTL_ERR_ARG, "ctl_set_values: the mass matrix has no time level");
        h->h_M.assign(values, values + nnz);
        cudaFree(h->d_M_full);          // rebuilt on the next ctl_objective
        h->d_M_full = nullptr;
    } else if (which == CTL_MAT_K || which == CTL_MAT_KT) {
        auto &dst = (which == CTL_MAT_K) ? h->h_K : h->h_KT;
        if (level == -1) {
            dst.assign(1, std::vector<double>(values, values + nnz));
        } else {
            if ((int)dst.size() != h->cfg.n_t) {
                // switching from "all levels" to per-level storage: replicate what is there
                std::vector<double> proto = dst.size() == 1 ? dst[0] : std::vector<double>(nnz, 0.0);
                dst.assign(h->cfg.n_t, proto);
            }
            dst[level].assign(values, values + nnz);
        }
    } else {
        CTL_CHECK(false, CTL_ERR_ARG, "ctl_set_values: unknown matrix id");
    }
    ctl_lift_invalidate(h);             // the lifting reads M and K: rebuilt on the next ctl_lift_bc
    h->assembled = false;
    return CTL_OK;
}

int ctl_set_block_size(ctl_handle h, int32_t bs)
{
    CTL_CHECK(h, CTL_ERR_ARG, "ctl_set_block_size: null handle");
    CTL_CHECK(bs >= 1 && bs <= 3, CTL_ERR_ARG, "ctl_set_block_size: the block size must be 1, 2 or 3");
    CTL_CHECK(h->n % bs == 0, CTL_ERR_ARG, "ctl_set_block_size: n is not a multiple of the block size");
    CTL_CHECK(bs == 1 || h->cfg.world == 1, CTL_ERR_ARG, "ctl_set_block_size: block-scalar sweeps run on one GPU (world 1)");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    h->block_size = bs;
    ctl_pc_free(h);                     // set up again with the new block size
    return CTL_OK;
}

int ctl_set_bc(ctl_handle h, const int32_t *dofs, int32_t count)
{
    CTL_CHECK(h && (dofs || count == 0) && count >= 0, CTL_ERR_ARG, "ctl_set_bc: bad argument");
    h->h_bc.assign(dofs, dofs + count);
    std::fill(h->h_bcmask.begin(), h->h_bcmask.end(), 0);
    for (int i = 0; i < count; ++i) {
        CTL_CHECK(dofs[i] >= 0 && dofs[i] < h->n, CTL_ERR_ARG, "ctl_set_bc: dof out of range");
        h->h_bcmask[dofs[i]] = 1;
    }
    ctl_lift_invalidate(h);
    h->assembled = false;
    return CTL_OK;
}

// Build the local row block (pattern part), once per pattern.
static int build_local_pattern(ctl_handle_s *h)
{
    const int rb = h->row_begin, nl = h->n_loc;
    const std::vector<int> &ip = h->h_indptr, &ix = h->h_indices;
    // ghost columns, sorted by global id (= grouped by owner for a contiguous partition)
    std::vector<int> ghosts;
    for (int r = rb; r < rb + nl; ++r)
        for (int k = ip[r]; k < ip[r + 1]; ++k)
            if (ix[k] < rb || ix[k] >= rb + nl) ghosts.push_back(ix[k]);
    std::sort(ghosts.begin(), ghosts.end());
    ghosts.erase(std::unique(ghosts.begin(), ghosts.end()), ghosts.end());
    h->halo_global = ghosts;
    h->n_halo = (int)ghosts.size();
    HostCSR &L = h->loc;
    L.n_rows = nl;
    L.n_cols = nl + h->n_halo;
    L.indptr.assign(nl + 1, 0);
    const int64_t nnz_loc = ip[rb + nl] - ip[rb];
    L.indices.resize(nnz_loc);
    h->loc_entry.resize(nnz_loc);
    h->loc_tperm.resize(nnz_loc);
    int64_t p = 0;
    for (int r = 0; r < nl; ++r) {
        const int g = rb + r;
        for (int k = ip[g]; k < ip[g + 1]; ++k, ++p) {
            const int c = ix[k];
            int lc;
            if (c >= rb && c < rb + nl) lc = c - rb;
            else lc = nl + (int)(std::lower_bound(ghosts.begin(), ghosts.end(), c) - ghosts.begin());
            L.indices[p] = lc;
            h->loc_entry[p] = k;
            // entry (c, g) of the global pattern, for K^T on the same pattern
            const int *b = ix.data() + ip[c], *e = ix.data() + ip[c + 1];
            const int *f = std::lower_bound(b, e, g);
            h->loc_tperm[p] = (f != e && *f == g) ? (int)(f - ix.data()) : -1;
        }
        L.indptr[r + 1] = (int)p;
        h->max_row_len = std::max(h->max_row_len, ip[g + 1] - ip[g]);
    }
    {   // gather chunk with the fewest padding slots over all rows (ties: the larger chunk)
        const int cand[4] = {4, 5, 7, 8};
        long best = -1;
        for (int c : cand) {
            long slots = 0;
            for (int r = 0; r < nl; ++r) {
                const int len = L.indptr[r + 1] - L.indptr[r];
                slots += (long)((len + c - 1) / c) * c;
            }
            if (best < 0 || slots <= best) {
                best = slots;
                h->gather_chunk = c;
            }
        }
    }
    // note: local column order within a row is no longer sorted when ghosts precede owned
    // columns globally; the kernels do not rely on sorted columns.
    return CTL_OK;
}

int ctl_assemble(ctl_handle h)
{
    CTL_CHECK(h, CTL_ERR_ARG, "ctl_assemble: null handle");
    CTL_CHECK(!h->h_indptr.empty(), CTL_ERR_STATE, "ctl_assemble: no pattern");
    CTL_CHECK(!h->h_M.empty(), CTL_ERR_STATE, "ctl_assemble: mass matrix values missing");
    CTL_CHECK(!h->h_K.empty(), CTL_ERR_STATE, "ctl_assemble: K values missing");
    CTL_CHECK(h->h_KT.empty() || h->h_KT.size() == h->h_K.size(), CTL_ERR_STATE,
              "ctl_assemble: K and K^T must both be per-level or both time independent");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    if (h->loc.n_rows == 0) {
        CTL_TRY(build_local_pattern(h));
        CTL_TRY(ctl_upload(h, &h->d_indptr, h->loc.indptr.data(), h->loc.indptr.size()));
        CTL_TRY(ctl_upload(h, &h->d_indices, h->loc.indices.data(), h->loc.indices.size()));
    }
    const int nl = h->n_loc, rb = h->row_begin;
    const int64_t nnz = h->loc.nnz();
    const bool have_kt = !h->h_KT.empty();
    if (!have_kt)
        for (int64_t p = 0; p < nnz; ++p)
            CTL_CHECK(h->loc_tperm[p] >= 0, CTL_ERR_ARG,
                      "ctl_assemble: pattern is not structurally symmetric; supply CTL_MAT_KT");
    // Dirichlet mask on local rows (owned + ghost)
    std::vector<uint8_t> mask(nl + h->n_halo);
    for (int r = 0; r < nl; ++r) mask[r] = h->h_bcmask[rb + r];
    for (int g = 0; g < h->n_halo; ++g) mask[nl + g] = h->h_bcmask[h->halo_global[g]];
    CTL_TRY(ctl_upload(h, &h->d_bcmask, mask.data(), mask.size()));
    {
        std::vector<int> rows;
        for (int r = 0; r < nl; ++r)
            if (mask[r]) rows.push_back(r);
        h->n_bc_all = (int)rows.size();
        CTL_TRY(ctl_upload(h, &h->d_bc_rows_all, rows.data(), rows.size()));
    }
    auto colmask = [&](int64_t p) { return mask[h->loc.indices[p]] != 0; };

    std::vector<double> buf(nnz);
    for (int64_t p = 0; p < nnz; ++p) buf[p] = colmask(p) ? 0.0 : h->h_M[h->loc_entry[p]];
    CTL_TRY(ctl_upload(h, &h->d_M, buf.data(), buf.size()));

    if (h->d_KT && h->d_KT != h->d_K) cudaFree(h->d_KT);
    h->d_KT = nullptr;
    h->per_level = h->h_K.size() > 1;
    auto kt_value = [&](int level, int64_t p) {
        return have_kt ? h->h_KT[level][h->loc_entry[p]] : h->h_K[level][h->loc_tperm[p]];
    };
    if (!h->per_level) {
        bool sym = true;
        std::vector<double> bt(nnz);
        for (int64_t p = 0; p < nnz; ++p) {
            const bool z = colmask(p);
            buf[p] = z ? 0.0 : h->h_K[0][h->loc_entry[p]];
            bt[p] = z ? 0.0 : kt_value(0, p);
            sym = sym && (buf[p] == bt[p]);
        }
        CTL_TRY(ctl_upload(h, &h->d_K, buf.data(), buf.size()));
        h->k_symmetric = sym;
        if (sym) h->d_KT = h->d_K;
        else CTL_TRY(ctl_upload(h, &h->d_KT, bt.data(), bt.size()));
    } else {
        // panels [nnz][ld]: column j of the K panel multiplies column j of X_v, i.e. level
        // j+1 for CN (block j holds v_{j+1}) and level j for BE; the K^T panel holds level j
        const int ld = h->ld, N = h->N;
        std::vector<double> pk((size_t)nnz * ld, 0.0), pt((size_t)nnz * ld, 0.0);
        for (int64_t p = 0; p < nnz; ++p) {
            if (colmask(p)) continue;
            for (int j = 0; j < N; ++j) {
                const int lv = h->cfg.CN ? j + 1 : j;
                pk[(size_t)p * ld + j] = h->h_K[lv][h->loc_entry[p]];
                pt[(size_t)p * ld + j] = kt_value(j, p);
            }
        }
        CTL_TRY(ctl_upload(h, &h->d_K, pk.data(), pk.size()));
        CTL_TRY(ctl_upload(h, &h->d_KT, pt.data(), pt.size()));
        h->k_symmetric = false;
    }
    if (h->n_halo > 0 && !h->d_halo) {
        CTL_CUDA(cudaMalloc((void **)&h->d_halo, (size_t)2 * h->n_halo * h->ld * sizeof(double)));
        CTL_CUDA(cudaMemsetAsync(h->d_halo, 0, (size_t)2 * h->n_halo * h->ld * sizeof(double), h->stream));
    }
    CTL_TRY(ctl_pc_invalidate(h));
    h->assembled = true;
    return CTL_OK;
}

int32_t ctl_n_blocks(ctl_handle h) { return h ? h->N : 0; }
int32_t ctl_ld(ctl_handle h) { return h ? h->ld : 0; }
int32_t ctl_n_local(ctl_handle h) { return h ? h->n_loc : 0; }
int32_t ctl_row_begin(ctl_handle h) { return h ? h->row_begin : 0; }
int64_t ctl_vec_len(ctl_handle h, int layout)
{
    if (!h) return 0;
    return layout == CTL_LAYOUT_TIME_FASTEST ? h->vec_len() : 2ll * h->N * h->n_loc;
}
int64_t ctl_kernel_launches(ctl_handle h) { return h ? h->launches : 0; }

int ctl_convert_layout(ctl_handle h, const double *src, int src_layout, double *dst, int dst_layout)
{
    CTL_CHECK(h && src && dst, CTL_ERR_ARG, "ctl_convert_layout: null argument");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    if (src_layout == dst_layout) {
        CTL_CUDA(cudaMemcpyAsync(dst, src, ctl_vec_len(h, src_layout) * sizeof(double),
                                 cudaMemcpyDeviceToDevice, h->stream));
        return CTL_OK;
    }
    if (src_layout == CTL_LAYOUT_BLOCK_MAJOR) return ctl_to_tf(h, src, dst);
    return ctl_to_bm(h, src, dst);
}

int ctl_kkt_apply(ctl_handle h, const double *x, double *y, int layout)
{
    CTL_CHECK(h && x && y, CTL_ERR_ARG, "ctl_kkt_apply: null argument");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    if (layout == CTL_LAYOUT_TIME_FASTEST) return ctl_kkt_apply_tf(h, x, y);
    return with_tf(h, layout, {x, nullptr}, y,
                   [&](const double *xt, double *yt) { return ctl_kkt_apply_tf(h, xt, yt); });
}

int ctl_time_kkt_apply(ctl_handle h, const double *x_tf, double *y_tf, int reps, float *ms)
{
    CTL_CHECK(h && x_tf && y_tf && ms && reps > 0, CTL_ERR_ARG, "ctl_time_kkt_apply: bad argument");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    EventPair ev;
    CTL_TRY(ev.create(h));
    CTL_CUDA(cudaEventRecord(ev.begin, h->stream));
    int rc = CTL_OK;
    for (int i = 0; i < reps && rc == CTL_OK; ++i) rc = ctl_kkt_apply_tf(h, x_tf, y_tf);
    CTL_CUDA(cudaEventRecord(ev.end, h->stream));
    CTL_CUDA(cudaEventSynchronize(ev.end));
    float t = 0;
    CTL_CUDA(cudaEventElapsedTime(&t, ev.begin, ev.end));
    *ms = t / reps;
    return rc;
}

}  // extern "C"
