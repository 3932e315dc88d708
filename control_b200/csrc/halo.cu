// Device-initiated halo exchange, host side (see halo.cuh for the protocol) and the distributed AMG hierarchy.
//
// Why three slots are enough.  Let kernel k of a rank push exchange k of a space and kernel k+1 gather it.  A can
// start kernel k+1 only after its own kernel k, and its boundary rows complete in it only after B's push k has
// arrived, i.e. after B's kernel k has STARTED (the push warps run first).  So when A pushes exchange k+1 (slot (k+1) % 3), B is at
// least inside kernel k, whose regular CTAs may still read slot (k-1) % 3 and will read slot k % 3 next: both
// differ from the slot being written.  A cannot push exchange k+2 before B's push k+1 arrived, i.e. before B's
// kernel k has completed, which ends B's last read of slot (k-1) % 3 = (k+2) % 3.
// Across sweep replays the static counters restart: halo_epoch_begin puts a barrier in between.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <map>

#include "comm.cuh"
#include "halo_host.cuh"
#include "pc.cuh"

// ---------------------------------------------------------------------------------------------------------
// geometry (halo_geom.h) -> device arrays of this rank's send side
// ---------------------------------------------------------------------------------------------------------
HaloSpace::~HaloSpace()
{
    cudaFree(d_rows);
    cudaFree(d_chunks);
    cudaFree(d_pos);
}

int halo_space_upload(ctl_handle_s *h, const std::shared_ptr<HaloGeom> &g, std::shared_ptr<HaloSpace> &out)
{
    auto sp = std::make_shared<HaloSpace>();
    sp->g = g;
    const std::vector<HaloGeom::Chunk> &mine = g->chunks[g->me];
    std::vector<PushChunk> pc(mine.size());
    std::vector<int> pos;
    int pairs = 0;
    for (size_t c = 0; c < mine.size(); ++c) {
        pc[c].start = mine[c].start;
        pc[c].count = mine[c].count;
        pc[c].dst_begin = pairs;
        pc[c].n_dst = (int)mine[c].dst.size();
        CTL_CHECK(pc[c].n_dst <= 32, CTL_ERR_ARG, "halo: a row is gathered by more than 32 ranks");
        pos.insert(pos.end(), mine[c].pos.begin(), mine[c].pos.end());
        pairs += pc[c].n_dst;
    }
    sp->n_pairs = pairs;
    CTL_TRY(ctl_upload(h, &sp->d_rows, g->send_rows[g->me].data(), g->send_rows[g->me].size()));
    if (!pc.empty()) {
        CTL_CUDA(cudaMalloc((void **)&sp->d_chunks, pc.size() * sizeof(PushChunk)));
        CTL_CUDA(cudaMemcpy(sp->d_chunks, pc.data(), pc.size() * sizeof(PushChunk), cudaMemcpyHostToDevice));
    }
    CTL_TRY(ctl_upload(h, &sp->d_pos, pos.data(), pos.size()));
    out = sp;
    return CTL_OK;
}

// ---------------------------------------------------------------------------------------------------------
// arena
// ---------------------------------------------------------------------------------------------------------
static size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

void halo_arena_free(ctl_handle_s *h, HaloArena &a)
{
    if (h->comm) {
        std::vector<HaloPlan *> &live = h->comm->plans;
        for (HaloArena::Inst &i : a.inst) live.erase(std::remove(live.begin(), live.end(), i.plan.get()), live.end());
    }
    for (HaloArena::Inst &i : a.inst) cudaFree(i.d_dsts);
    for (void *p : a.opened) cudaIpcCloseMemHandle(p);
    cudaFree(a.base);
    a = HaloArena();
}

HaloPlan *halo_arena_add(ctl_handle_s *h, HaloArena &a, const std::shared_ptr<HaloSpace> &sp)
{
    const HaloGeom &g = *sp->g;
    const int world = g.world;
    if (a.cursor.empty()) a.cursor.assign(world, 0);
    HaloArena::Inst in;
    in.sp = sp;
    in.plan.reset(new HaloPlan());
    in.slot_off.resize(world);
    for (int r = 0; r < world; ++r) {
        in.slot_off[r] = a.cursor[r];
        a.cursor[r] += align256((size_t)3 * g.stride(r) * sizeof(ulonglong2));
    }
    HaloPlan &p = *in.plan;
    p.n_own = g.n_own();
    p.n_ghost = g.n_ghost();
    p.replicate = g.replicate;
    p.d_chunks = sp->d_chunks;
    p.d_rows = sp->d_rows;
    p.n_chunks = (int)g.chunks[g.me].size();
    p.stride = g.stride(g.me);
    a.inst.push_back(std::move(in));
    return a.inst.back().plan.get();
}

int halo_arena_finalize(ctl_handle_s *h, HaloArena &a)
{
    CommState &c = *h->comm;
    const int world = c.world, me = c.rank;
    if (a.cursor.empty()) a.cursor.assign(world, 0);
    const size_t bytes = std::max<size_t>(a.cursor[me], 256);
    CTL_CUDA(cudaMalloc((void **)&a.base, bytes));
    CTL_CUDA(cudaMemset(a.base, 0, bytes));
    // IPC handles travel through the communicator; every rank reports whether it could open all of them, and all
    // ranks take the same exit
    cudaIpcMemHandle_t mine;
    memset(&mine, 0, sizeof(mine));
    int ok = cudaIpcGetMemHandle(&mine, a.base) == cudaSuccess ? 1 : 0;
    if (!ok) cudaGetLastError();
    cudaIpcMemHandle_t *d_all = nullptr;
    int *d_ok = nullptr;
    CTL_CUDA(cudaMalloc((void **)&d_all, world * sizeof(cudaIpcMemHandle_t)));
    CTL_CUDA(cudaMalloc((void **)&d_ok, sizeof(int)));
    int rc = CTL_OK;
    std::vector<cudaIpcMemHandle_t> all(world);
    do {
        if (cudaMemcpy(d_all + me, &mine, sizeof(mine), cudaMemcpyHostToDevice) != cudaSuccess) ok = 0;
        if (ncclAllGather(d_all + me, d_all, sizeof(mine), ncclChar, c.comm, h->stream) != ncclSuccess) {
            rc = CTL_ERR_NCCL;
            break;
        }
        if (cudaStreamSynchronize(h->stream) != cudaSuccess ||
            cudaMemcpy(all.data(), d_all, world * sizeof(mine), cudaMemcpyDeviceToHost) != cudaSuccess)
            ok = 0;
        a.peer_base.assign(world, nullptr);
        a.peer_base[me] = a.base;
        for (int r = 0; r < world && ok; ++r) {
            if (r == me) continue;
            void *p = nullptr;
            if (cudaIpcOpenMemHandle(&p, all[r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                cudaGetLastError();
                ok = 0;
                break;
            }
            a.opened.push_back(p);
            a.peer_base[r] = (char *)p;
        }
        if (cudaMemcpy(d_ok, &ok, sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess ||
            ncclAllReduce(d_ok, d_ok, 1, ncclInt, ncclMin, c.comm, h->stream) != ncclSuccess ||
            cudaStreamSynchronize(h->stream) != cudaSuccess ||
            cudaMemcpy(&ok, d_ok, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess)
            rc = CTL_ERR_NCCL;
    } while (0);
    cudaFree(d_all);
    cudaFree(d_ok);
    if (rc != CTL_OK) {
        ctl_set_error(h, "halo arena: exchanging the IPC handles failed");
        return rc;
    }
    CTL_CHECK(ok == 1, CTL_ERR_CUDA,
              "halo arena: CUDA IPC is not available between the ranks (peer access over NVLink is required)");
    for (HaloArena::Inst &in : a.inst) {
        const HaloGeom &sp = *in.sp->g;
        HaloPlan &p = *in.plan;
        p.slots = (ulonglong2 *)(a.base + in.slot_off[me]);
        std::vector<PushDst> dsts;
        const std::vector<HaloGeom::Chunk> &mine_chunks = sp.chunks[me];
        int pair = 0;
        for (const HaloGeom::Chunk &ch : mine_chunks)
            for (size_t d = 0; d < ch.dst.size(); ++d, ++pair) {
                const int r = ch.dst[d];
                PushDst t;
                t.base = (ulonglong2 *)(a.peer_base[r] + in.slot_off[r]);
                t.stride = sp.stride(r);
                t.pos = in.sp->d_pos + (size_t)pair * 32;
                dsts.push_back(t);
            }
        if (!dsts.empty()) {
            CTL_CUDA(cudaMalloc((void **)&in.d_dsts, dsts.size() * sizeof(PushDst)));
            CTL_CUDA(cudaMemcpy(in.d_dsts, dsts.data(), dsts.size() * sizeof(PushDst), cudaMemcpyHostToDevice));
        }
        p.d_dsts = in.d_dsts;
        c.plans.push_back(&p);
    }
    a.finalized = true;
    return CTL_OK;
}

// ---------------------------------------------------------------------------------------------------------
// plan instances
// ---------------------------------------------------------------------------------------------------------
HaloCtx halo_ctx(const ctl_handle_s *h)
{
    HaloCtx c;
    if (h->comm && h->comm->d_epoch) {
        c.epoch = h->comm->d_epoch;
        c.err = h->comm->d_err;
        c.max_spins = h->comm->max_spins;
        static const int early = [] {
            const char *e = getenv("CTL_MP_EARLY_WAIT");
            return (e && e[0] == '1') ? 1 : 0;
        }();
        c.early_wait = early;
    }
    return c;
}

HaloPush halo_push(HaloPlan *p)
{
    HaloPush q;
    if (!p) return q;
    q.chunks = p->d_chunks;
    q.dsts = p->d_dsts;
    q.rows = p->d_rows;
    q.n_chunks = p->n_chunks;
    q.slot = (int)(p->idx % 3);
    q.idx1 = p->idx + 1;
    q.all_rows = p->replicate ? 1 : 0;
    p->idx++;
    return q;
}

const ulonglong2 *halo_ll(const HaloPlan *p) { return p->slots + (long long)((p->idx + 2) % 3) * p->stride; }
unsigned halo_idx1(const HaloPlan *p) { return p->idx; }      // the last exchange had index idx - 1

namespace {

__global__ void epoch_bump_kernel(unsigned long long *epoch) { *epoch += 1ull; }
// A complete kernel boundary behind the bump.  The sweep kernels read the epoch word BEFORE they wait for their
// predecessor (sell.cu, kernel_prologue); a kernel launched with the programmatic attribute right behind the bump could
// do so before the bump's store is visible.  This one is launched without the attribute: it starts after the bump has
// completed and its store has been flushed, and everything launched later starts later still.
__global__ void epoch_fence_kernel() {}

// boundary rows of an existing vector: push warps only
__global__ void __launch_bounds__(128) halo_push_kernel(const double *__restrict__ x, const HaloCtx ctx, const HaloPush push)
{
    pdl_sync();
    const int ci = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (ci >= push.n_chunks) return;
    const PushChunk ch = push.chunks[ci];
    if (lane >= ch.count) return;
    const unsigned seq = halo_epoch_bits(ctx) | push.idx1;
    const double v = x[push.rows[ch.start + lane]];
    for (int d = 0; d < ch.n_dst; ++d) {
        const PushDst t = push.dsts[ch.dst_begin + d];
        halo_ll_store(t.base + (long long)push.slot * t.stride + t.pos[lane], v, seq);
    }
}

__global__ void __launch_bounds__(128) halo_unpack_kernel(const ulonglong2 *slot, unsigned idx1, const HaloCtx ctx, double *dst, int n)
{
    pdl_sync();
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i < n) dst[i] = halo_ll_read(slot + i, halo_epoch_bits(ctx) | idx1, ctx);
}

}  // namespace

int halo_exchange_now(ctl_handle_s *h, HaloPlan *p, const double *x)
{
    if (!p) return CTL_OK;
    const HaloPush push = halo_push(p);
    if (push.n_chunks == 0) return CTL_OK;
    pdl_launch(h, (push.n_chunks + 3) / 4, 128, halo_push_kernel, x, halo_ctx(h), push);
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

int halo_unpack(ctl_handle_s *h, HaloPlan *p, double *dst)
{
    if (!p || p->n_ghost == 0) return CTL_OK;
    pdl_launch(h, (p->n_ghost + 127) / 128, 128, halo_unpack_kernel, halo_ll(p), halo_idx1(p), halo_ctx(h), dst, p->n_ghost);
    h->launches++;
    CTL_CUDA(cudaGetLastError());
    return CTL_OK;
}

int halo_epoch_begin(ctl_handle_s *h)
{
    if (!h->comm || h->comm->plans.empty()) return CTL_OK;
    CommState &c = *h->comm;
    CTL_NCCL(ncclAllReduce(c.d_barrier, c.d_barrier, 1, ncclInt, ncclMax, c.comm, h->stream));
    epoch_bump_kernel<<<1, 1, 0, h->stream>>>(c.d_epoch);
    epoch_fence_kernel<<<1, 1, 0, h->stream>>>();
    h->launches += 2;
    CTL_CUDA(cudaGetLastError());
    for (HaloPlan *p : c.plans) p->idx = 0;
    return CTL_OK;
}

// ---------------------------------------------------------------------------------------------------------
// distributed hierarchy: halo_geom.h::amg_distribute_host decides and extracts, this uploads
// ---------------------------------------------------------------------------------------------------------
int amg_level_vectors(ctl_handle_s *h, AmgLevelDev &L, int level);      // amg.cu

static void finish_matrix(const HostCSR &, int n_own_cols, SellMat &M)
{
    if (n_own_cols > 0) M.n_own = n_own_cols;      // columns behind it are ghosts
}

int amg_build_distributed(ctl_handle_s *h, const AmgParams &p, const std::shared_ptr<SellPattern> &fine_pattern,
                          AmgHierarchyDev &H)
{
    CTL_CHECK(h->pc && h->pc->mesh_space, CTL_ERR_STATE, "amg_build: the exchange geometry of the mesh is missing");
    CTL_CHECK(fine_pattern != nullptr, CTL_ERR_ARG, "amg_build: level 0 needs the mesh pattern");
    CTL_CHECK(p.nu >= 3 && (p.nu_fine == 0 || p.nu_fine >= 3), CTL_ERR_ARG,
              "amg_build: smoother degrees below 3 are not supported on several GPUs");
    CTL_CHECK(p.acc_lo <= 0.0, CTL_ERR_ARG, "amg_build: accelerated cycles are not supported on several GPUs");
    PcState &st = *h->pc;
    const int world = h->cfg.world, me = h->cfg.rank;
    const int nl = (int)H.host.size();
    // A coarse level with fewer matrix entries per rank than this (and everything below it) is replicated.  Measured
    // at C2 on 2 GPUs (profiles/r02_multi_gpu.txt): a product with the 2.3 M entries of the first Galerkin level
    // takes ~5 us on one GPU and an exchange puts ~5 us of NVLink latency on the critical path, so distributing
    // that level costs more than it saves (inner solve 1.12 ms against 0.70 ms with only the fine level
    // distributed); a level pays once its products are stream bound (3-D: 18.5 M entries on the first level of C3).
    int64_t rep_nnz = 2000000;
    if (const char *e = getenv("CTL_AMG_REP_NNZ")) rep_nnz = std::max(1ll, atoll(e));
    DistHierarchy D;
    amg_distribute_host(world, me, H.host, rep_nnz, st.mesh_space->g, D);
    CTL_CHECK(D.part[0][me] == h->row_begin && D.part[0][me + 1] - D.part[0][me] == h->n_loc, CTL_ERR_STATE,
              "amg_build: level-0 partition differs from the handle's");
    CTL_CHECK(st.mesh_space->g->ghosts[me] == h->halo_global, CTL_ERR_STATE, "amg_build: mesh ghosts differ from the handle's");
    std::shared_ptr<HaloSpace> sp_r0;
    CTL_TRY(halo_space_upload(h, D.space_r0, sp_r0));
    H.spaces.push_back(sp_r0);
    for (int l = 0; l < nl; ++l) {
        AmgLevelHost &Lh = H.host[l];
        DistLevel &Dl = D.levels[l];
        AmgLevelDev &Ld = H.dev[l];
        Ld.distributed = Dl.distributed;
        Ld.n = Dl.n;
        Ld.n_ghost = Dl.n_ghost;
        Ld.rho = Lh.rho;
        std::shared_ptr<HaloSpace> sp;
        if (l == 0) sp = st.mesh_space;
        else if (Dl.space) {
            CTL_TRY(halo_space_upload(h, Dl.space, sp));
            H.spaces.push_back(sp);
        }
        if (Dl.distributed) {
            Ld.px = l == 0 ? st.px0 : halo_arena_add(h, st.arena, sp);
            Ld.pb = l == 0 ? st.pb0 : halo_arena_add(h, st.arena, sp);
            if (l == 0) Ld.pr = halo_arena_add(h, st.arena, sp_r0);
        } else if (l == D.L_rep) {
            Ld.prep = halo_arena_add(h, st.arena, sp);
        }
        if (l == 0) {
            std::vector<double> lv(h->loc_entry.size());
            for (size_t q = 0; q < lv.size(); ++q) lv[q] = Lh.A.values[h->loc_entry[q]];
            CTL_TRY(sell_set_values(h, fine_pattern, lv.data(), Ld.A));
            finish_matrix(h->loc, h->n_loc, Ld.A);
        } else {
            CTL_TRY(sell_from_csr(h, Dl.A, Ld.A));
            finish_matrix(Dl.A, Dl.A_own, Ld.A);
        }
        CTL_TRY(ctl_upload(h, &Ld.dinv, Dl.dinv.data(), Dl.dinv.size()));
        CTL_TRY(amg_level_vectors(h, Ld, l));
        if (l + 1 < nl) {
            CTL_TRY(sell_from_csr(h, Dl.P, Ld.P));
            finish_matrix(Dl.P, Dl.P_own, Ld.P);
            CTL_TRY(sell_from_csr(h, Dl.R, Ld.R));
            finish_matrix(Dl.R, Dl.R_own, Ld.R);
        } else if (!Dl.Ainv.empty()) {
            CTL_TRY(dense_inverse_upload(h, Dl.Ainv, Dl.n, &Ld.Ainv, &Ld.Ainv_ld));
        } else if (Dl.coarse_inverse) {
            CTL_CHECK(Dl.A.n_rows == Dl.n && Dl.A.n_cols == Dl.n, CTL_ERR_STATE, "amg_build: the level with the dense inverse must be replicated");
            CTL_TRY(dense_inverse_device(h, Dl.A, Dl.coarse_shift, &Ld.Ainv, &Ld.Ainv_ld));
        }
    }
    return CTL_OK;
}
