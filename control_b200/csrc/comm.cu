// Multi-GPU plumbing: one process per GPU, rows of the spatial mesh partitioned in
// contiguous blocks (PETSc's ownership split, as the reference's MPIAIJ matrices are
// distributed: preconditioner/preconditioner.py:706-722 sizes the shell Mat ((n_local,
// N_global), ...)).  Every rank keeps ALL N time columns of its rows, so the time axis
// never communicates.  Two collectives over NCCL / NVLink, both enqueued on the handle's
// stream (and therefore capturable into the sweep CUDA graph):
//   * halo exchange of boundary rows before a sparse product (what PETSc's VecScatter
//     does inside MatMult_MPIAIJ): rows x ld doubles per neighbour for the time-batched
//     kernels, one double per row for the single-column sweep kernels;
//   * all-reduce of a handful of doubles per Krylov iteration (VecMDot / VecNorm) and of
//     the restricted coarse right-hand side inside an AMG cycle (coarse levels are
//     replicated on every rank).
// The exchange plan needs no communication: every rank holds the global sparsity pattern
// and derives, deterministically, both what it needs and what each peer needs from it.
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "comm.cuh"

void ctl_comm_free(ctl_handle_s *h)
{
    if (!h->comm) return;
    CommState &c = *h->comm;
    cudaFree(c.d_epoch);
    cudaFree(c.d_err);
    cudaFree(c.d_barrier);
    if (c.comm) ncclCommDestroy(c.comm);
    h->comm.reset();
}

namespace {

// gather rows of a [rows x width] row-major array: out[i, :] = in[rows[i], :]
__global__ void pack_rows_kernel(const double *__restrict__ in, const int *__restrict__ rows, int n_rows, int width,
                                 double *__restrict__ out)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)n_rows * width) return;
    const int i = (int)(t / width), j = (int)(t % width);
    out[t] = in[(size_t)rows[i] * width + j];
}

}  // namespace

int exchange_plan_build(ctl_handle_s *h, const int *ip, const int *ix, int n_rows, int n_cols, int world, int me,
                        ExchangePlan &P)
{
    exchange_lists(ip, ix, n_rows, n_cols, world, me, P);
    P.n_send = (int)P.send_rows.size();
    CTL_TRY(ctl_upload(h, &P.d_send_rows, P.send_rows.data(), P.send_rows.size()));
    if (P.n_send > 0)
        CTL_CUDA(cudaMalloc((void **)&P.d_sendbuf, (size_t)2 * P.n_send * h->ld * sizeof(double)));
    return CTL_OK;
}

int exchange_plan_run(ctl_handle_s *h, ncclComm_t comm, const ExchangePlan &P, const double *x_tf,
                      size_t panel_stride, int panels, double *ghost)
{
    const int ld = h->ld;
    const size_t n_ghost = P.ghosts.size();
    for (int p = 0; p < panels; ++p) {
        if (P.n_send == 0) break;
        const int64_t total = (int64_t)P.n_send * ld;
        pack_rows_kernel<<<ceil_div(total, 256), 256, 0, h->stream>>>(x_tf + p * panel_stride, P.d_send_rows, P.n_send,
                                                                     ld, P.d_sendbuf + (size_t)p * P.n_send * ld);
        h->launches++;
    }
    CTL_CUDA(cudaGetLastError());
    CTL_NCCL(ncclGroupStart());
    for (size_t i = 0; i < P.peers.size(); ++i) {
        for (int p = 0; p < panels; ++p) {
            if (P.send_cnt[i])
                CTL_NCCL(ncclSend(P.d_sendbuf + ((size_t)p * P.n_send + P.send_off[i]) * ld, (size_t)P.send_cnt[i] * ld,
                                  ncclDouble, P.peers[i], comm, h->stream));
            if (P.recv_cnt[i])
                CTL_NCCL(ncclRecv(ghost + ((size_t)p * n_ghost + P.recv_off[i]) * ld, (size_t)P.recv_cnt[i] * ld,
                                  ncclDouble, P.peers[i], comm, h->stream));
        }
    }
    CTL_NCCL(ncclGroupEnd());
    return CTL_OK;
}

// exchange `panels` time-fastest panels through the mesh pattern: ghost rows land in h->d_halo[p]
static int exchange_panels(ctl_handle_s *h, const double *x_tf, int panels)
{
    return exchange_plan_run(h, h->comm->comm, h->comm->mesh, x_tf, (size_t)h->n_loc * h->ld, panels, h->d_halo);
}

int ctl_halo_exchange(ctl_handle_s *h, const double *x_tf)
{
    if (!h->comm || h->n_halo == 0) return CTL_OK;
    return exchange_panels(h, x_tf, 2);
}

int ctl_halo_exchange_panel(ctl_handle_s *h, const double *panel_tf)
{
    if (!h->comm || h->n_halo == 0) return CTL_OK;
    return exchange_panels(h, panel_tf, 1);
}

// has a device-side wait of the sweep kernels given up (bounded spin, halo.cuh)?  Called by every public entry
// point that runs sweeps; the flag is cleared once reported.
int ctl_comm_check(ctl_handle_s *h)
{
    if (!h->comm || !h->comm->d_err) return CTL_OK;
    int err = 0;
    CTL_CUDA(cudaMemcpyAsync(&err, h->comm->d_err, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CTL_CUDA(cudaStreamSynchronize(h->stream));
    if (err != 0) {
        CTL_CUDA(cudaMemsetAsync(h->comm->d_err, 0, sizeof(int), h->stream));
        CTL_CHECK(false, CTL_ERR_NCCL, "halo exchange timed out waiting for a neighbour (CTL_HALO_TIMEOUT_MS)");
    }
    return CTL_OK;
}

int ctl_allreduce_sum(ctl_handle_s *h, double *dev, int count)
{
    if (!h->comm) return CTL_OK;
    CTL_NCCL(ncclAllReduce(dev, dev, (size_t)count, ncclDouble, ncclSum, h->comm->comm, h->stream));
    return CTL_OK;
}

extern "C" {

int ctl_comm_unique_id(void *id128)
{
    if (!id128) return CTL_ERR_ARG;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is expected to be 128 bytes");
    ncclUniqueId id;
    if (ncclGetUniqueId(&id) != ncclSuccess) return CTL_ERR_NCCL;
    memcpy(id128, &id, sizeof(id));
    return CTL_OK;
}

int ctl_comm_init(ctl_handle h, const void *id128)
{
    CTL_CHECK(h && id128, CTL_ERR_ARG, "ctl_comm_init: null argument");
    CTL_CHECK(h->cfg.world > 1, CTL_ERR_STATE, "ctl_comm_init: the handle was created with world = 1");
    CTL_CHECK(h->assembled, CTL_ERR_STATE, "ctl_comm_init: call ctl_assemble first");
    CTL_CUDA(cudaSetDevice(h->cfg.device));
    ctl_comm_free(h);
    h->comm = std::make_shared<CommState>();
    CommState &c = *h->comm;
    c.rank = h->cfg.rank;
    c.world = h->cfg.world;
    ncclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    CTL_NCCL(ncclCommInitRank(&c.comm, c.world, id, c.rank));
    CTL_TRY(exchange_plan_build(h, h->h_indptr.data(), h->h_indices.data(), h->n, h->n, c.world, c.rank, c.mesh));
    CTL_CHECK(c.mesh.ghosts == h->halo_global, CTL_ERR_STATE, "ctl_comm_init: exchange plan and local pattern disagree");
    // device words of the in-kernel exchange (halo.cu)
    CTL_CUDA(cudaMalloc((void **)&c.d_epoch, sizeof(unsigned long long)));
    CTL_CUDA(cudaMemset(c.d_epoch, 0, sizeof(unsigned long long)));
    CTL_CUDA(cudaMalloc((void **)&c.d_err, sizeof(int)));
    CTL_CUDA(cudaMemset(c.d_err, 0, sizeof(int)));
    CTL_CUDA(cudaMalloc((void **)&c.d_barrier, sizeof(int)));
    CTL_CUDA(cudaMemset(c.d_barrier, 0, sizeof(int)));
    long long ms = 20000;
    if (const char *e = getenv("CTL_HALO_TIMEOUT_MS")) ms = std::max(1ll, atoll(e));
    c.max_spins = ms * 2000;      // one spin is a 20 ns sleep plus an L2 read: about half a microsecond
    return CTL_OK;
}

}  // extern "C"
