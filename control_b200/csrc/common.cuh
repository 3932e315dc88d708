// Internal declarations shared by the translation units of libctl_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <array>
#include <cstdio>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/ctl_b200.h"

struct ctl_handle_s;

// ---------------------------------------------------------------- error plumbing
#define CTL_CUDA(call)                                                                     \
    do {                                                                                   \
        cudaError_t e__ = (call);                                                          \
        if (e__ != cudaSuccess) {                                                          \
            ctl_set_error(h, std::string(#call) + ": " + cudaGetErrorString(e__));         \
            return CTL_ERR_CUDA;                                                           \
        }                                                                                  \
    } while (0)

#define CTL_CHECK(cond, code, msg)                                                         \
    do {                                                                                   \
        if (!(cond)) {                                                                     \
            ctl_set_error(h, msg);                                                         \
            return (code);                                                                 \
        }                                                                                  \
    } while (0)

#define CTL_TRY(expr)                                                                      \
    do {                                                                                   \
        int rc__ = (expr);                                                                 \
        if (rc__ != CTL_OK) return rc__;                                                   \
    } while (0)

void ctl_set_error(ctl_handle_s *h, const std::string &msg);

// ---------------------------------------------------------------- host containers
struct HostCSR {
    int n_rows = 0, n_cols = 0;
    std::vector<int> indptr, indices;
    std::vector<double> values;
    int64_t nnz() const { return (int64_t)indices.size(); }
};

// ---------------------------------------------------------------- scoped device resources
// Each type below releases what it holds when it goes out of scope.  Outside this header no code destroys an event
// or touches a pool's free list (tests/test_source_rules.py).
class Scratch;

// Device vectors of one fixed length, reused last in, first out, and freed with the pool
class ScratchPool {
  public:
    ScratchPool() = default;
    ScratchPool(const ScratchPool &) = delete;
    ScratchPool &operator=(const ScratchPool &) = delete;
    ~ScratchPool()
    {
        for (double *p : free_) cudaFree(p);
    }
    void init(ctl_handle_s *h, int64_t len)   // h takes the error text of a failed allocation
    {
        h_ = h;
        len_ = len;
    }
    int take(Scratch *out);                   // *out (empty) holds one vector until it goes out of scope

  private:
    friend class Scratch;
    ctl_handle_s *h_ = nullptr;
    int64_t len_ = 0;
    std::vector<double *> free_;
};

// The lease of one vector of a ScratchPool: converts to the vector and gives it back when it goes out of scope
class Scratch {
  public:
    Scratch() = default;
    Scratch(Scratch &&o) noexcept : pool_(o.pool_), p_(o.p_) { o.p_ = nullptr; }
    ~Scratch()
    {
        if (p_) pool_->free_.push_back(p_);
    }
    operator double *() const { return p_; }

  private:
    friend class ScratchPool;
    ScratchPool *pool_ = nullptr;
    double *p_ = nullptr;
};

inline int ScratchPool::take(Scratch *out)
{
    ctl_handle_s *h = h_;
    if (free_.empty()) {
        double *p = nullptr;
        CTL_CUDA(cudaMalloc((void **)&p, (size_t)len_ * sizeof(double)));
        free_.push_back(p);
    }
    out->pool_ = this;
    out->p_ = free_.back();
    free_.pop_back();
    return CTL_OK;
}

// Two events around a timed region, destroyed with the pair
struct EventPair {
    cudaEvent_t begin = nullptr, end = nullptr;
    EventPair() = default;
    EventPair(EventPair &&o) noexcept : begin(o.begin), end(o.end) { o.begin = o.end = nullptr; }
    ~EventPair()
    {
        if (begin) cudaEventDestroy(begin);
        if (end) cudaEventDestroy(end);
    }
    int create(ctl_handle_s *h)
    {
        CTL_CUDA(cudaEventCreate(&begin));
        CTL_CUDA(cudaEventCreate(&end));
        return CTL_OK;
    }
};

// A device array for the temporaries of one call, freed when it goes out of scope
template <typename T>
struct DeviceArray {
    T *p = nullptr;
    DeviceArray() = default;
    DeviceArray(const DeviceArray &) = delete;
    DeviceArray &operator=(const DeviceArray &) = delete;
    ~DeviceArray() { cudaFree(p); }
    cudaError_t alloc(size_t count) { return cudaMalloc((void **)&p, count * sizeof(T)); }
    operator T *() const { return p; }
};

// Runs fn on internal-layout copies of an entry point's device vectors, one vector of `pool` each: fn's i-th
// argument holds to_internal(in[i]) (nothing for a null in[i]), and when fn succeeds the last one is written to `out`
// (if set) with to_caller.  Each system passes its own layout conversions.
template <size_t K, class In, class Out, class F>
int with_internal(ScratchPool &pool, const double *const (&in)[K], double *out, In to_internal, Out to_caller, F fn)
{
    Scratch t[K];
    for (Scratch &s : t) CTL_TRY(pool.take(&s));
    std::array<double *, K> p;
    for (size_t i = 0; i < K; ++i) {
        p[i] = t[i];
        if (in[i]) CTL_TRY(to_internal(in[i], p[i]));
    }
    CTL_TRY(std::apply(fn, p));
    return out ? to_caller(p[K - 1], out) : CTL_OK;
}

// ---------------------------------------------------------------- the handle
struct ctl_handle_s {
    ctl_config cfg{};
    int N = 0;                 // time blocks
    int ld = 0;                // padded columns of the time-fastest layout
    int n = 0;                 // global spatial dofs
    int n_loc = 0;             // rows owned by this rank
    int row_begin = 0;
    int n_halo = 0;            // ghost rows appended behind the owned rows
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    int64_t launches = 0;
    bool assembled = false;
    int block_size = 1;        // ctl_set_block_size: interleaved components of the space, dof = block_size node + comp

    // host copies of what the caller handed over (global numbering)
    std::vector<int> h_indptr, h_indices;
    std::vector<double> h_M;
    std::vector<std::vector<double>> h_K;     // 1 (all levels) or n_t value arrays
    std::vector<std::vector<double>> h_KT;    // optional, same shape as h_K
    std::vector<int> h_bc;
    std::vector<int> h_tperm;                 // global entry (r,c) -> entry index of (c,r); built on demand (pc.cu)
    std::vector<uint8_t> h_bcmask;            // global rows

    // local (this rank's rows) CSR in local column numbering: owned columns first, ghosts after
    HostCSR loc;                              // values unused; pattern only
    std::vector<int64_t> loc_entry;           // local entry -> global CSR entry index
    std::vector<int> loc_tperm;               // local entry (r,c) -> global entry index of (c,r)
    std::vector<int> halo_global;             // global row id of each ghost row

    // device: shared pattern + value sets of the batched (time-fastest) kernels
    int *d_indptr = nullptr, *d_indices = nullptr;
    double *d_M = nullptr;      // BC columns zeroed
    double *d_M_full = nullptr; // no elimination; uploaded on first use (objective.cu)
    double *d_K = nullptr;      // scalar per entry (time independent) or panel [nnz x ld]
    double *d_KT = nullptr;     // may alias d_K (symmetric, time independent)
    bool per_level = false;
    int max_row_len = 0;        // longest local row (sizes the shared-memory staging)
    int gather_chunk = 4;       // entries per gather pass of the staged KKT apply (4, 5, 7 or 8: least padding)
    bool k_symmetric = false;
    uint8_t *d_bcmask = nullptr;   // local rows (owned + ghost)
    int *d_bc_rows_all = nullptr;  // list of constrained owned rows
    int n_bc_all = 0;
    double *d_halo = nullptr;      // ghost rows of the current SpMM input, [2][n_halo x ld]

    // reduction workspace (vec_ops.cu)
    double *d_red = nullptr, *h_red = nullptr;

    // scratch vectors (time-fastest, 2 * n_loc * ld doubles each, at least one)
    ScratchPool pool;

    // preconditioner, Krylov workspace, communicator: defined in their own units
    std::shared_ptr<struct PcState> pc;
    std::shared_ptr<struct KrylovState> ks;
    std::shared_ptr<struct CommState> comm;
    std::shared_ptr<struct LiftState> lift;   // boundary-column CSR of ctl_lift_bc (lift.cu); null = build on next use
    ctl_pc_callback pc_cb = nullptr;
    void *pc_cb_user = nullptr;

    int64_t vec_len() const { return 2ll * n_loc * ld; }
};

// ---------------------------------------------------------------- kernels / helpers (defined in .cu files)
// layout.cu
int ctl_to_tf(ctl_handle_s *h, const double *src_bm, double *dst_tf);
int ctl_to_bm(ctl_handle_s *h, const double *src_tf, double *dst_bm);
// kkt_apply.cu
int ctl_kkt_apply_tf(ctl_handle_s *h, const double *x_tf, double *y_tf);
// pc.cu: Preconditioner.apply on time-fastest vectors
int ctl_pc_apply_tf(ctl_handle_s *h, const double *b_tf, double *u_tf);
// stokes.cu: in place on one time-fastest panel, X[r, :] <- T_1^-1 (which = 1) / T_2^-1 (which = 2) X[r, :]
int ctl_panel_tinv(ctl_handle_s *h, double *X, int which, int n_rows);
// krylov.cu: MultiBlockSystem.solve on time-fastest vectors (u: initial guess in, solution out)
int ctl_solve_tf(ctl_handle_s *h, const double *b_tf, double *u_tf, const ctl_krylov_options *opts,
                 ctl_solve_result *result);

// unit-private state teardown / invalidation
void ctl_pc_free(ctl_handle_s *h);        // pc.cu
void ctl_comm_free(ctl_handle_s *h);      // comm.cu
int ctl_pc_invalidate(ctl_handle_s *h);   // pc.cu: matrices changed, rebuild on next setup
void ctl_lift_invalidate(ctl_handle_s *h);   // lift.cu: M, K or the Dirichlet dofs changed
// lift.cu: the constrained-velocity columns of the divergence matrix B (n_p x n_v host CSR, values before
// elimination; columns in the ctl_set_bc list of the velocity handle h), and b_1_0 -= T_2(tau B g) on them
int ctl_lift_div_setup(ctl_handle_s *h, const int32_t *B_indptr, const int32_t *B_indices, const double *B_values,
                       int n_p, std::shared_ptr<struct LiftState> *out);
int ctl_lift_div_apply(ctl_handle_s *h, const struct LiftState *S, const double *g, double *b10, int n_p);
// comm.cu
int ctl_halo_exchange(ctl_handle_s *h, const double *x_tf);            // both panels -> d_halo
int ctl_halo_exchange_panel(ctl_handle_s *h, const double *panel_tf);  // one panel -> d_halo[0]
int ctl_allreduce_sum(ctl_handle_s *h, double *dev, int count);
int ctl_comm_check(ctl_handle_s *h);                                   // peer-to-peer exchange timed out?

template <typename T>
int ctl_upload(ctl_handle_s *h, T **dst, const T *src, size_t count);

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

#include "pdl.cuh"

#ifdef __CUDACC__
template <typename... KArgs, typename... Args>
inline void pdl_launch(ctl_handle_s *h, int grid, int block, void (*kernel)(KArgs...), Args &&...args)
{
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.stream = h->stream;
    cudaLaunchAttribute at;
    at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &at;
    cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif
