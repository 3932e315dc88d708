// Communicator state shared by comm.cu (NCCL: time-batched halo panels, Krylov all-reduces) and halo.cu (the
// device-initiated exchange of the single-column sweep kernels).
#pragma once
#include <nccl.h>

#include <vector>

#include "common.cuh"
#include "exchange_plan.h"
#include "halo.cuh"

// NCCL exchange of time-fastest panels through a sparsity pattern (exchange_plan.h): the host lists, and the packed
// row list and send buffer on the device
struct ExchangePlan : ExchangeLists {
    int n_send = 0;
    int *d_send_rows = nullptr;           // send_rows on the device
    double *d_sendbuf = nullptr;          // [2][n_send x ld]
    ExchangePlan() = default;
    ExchangePlan(const ExchangePlan &) = delete;
    ExchangePlan &operator=(const ExchangePlan &) = delete;
    ~ExchangePlan()
    {
        cudaFree(d_send_rows);
        cudaFree(d_sendbuf);
    }
};

// the plan of the rows [row split of n_rows] of a global CSR pattern over the columns [column split of n_cols]
int exchange_plan_build(ctl_handle_s *h, const int *indptr, const int *indices, int n_rows, int n_cols, int world,
                        int rank, ExchangePlan &P);
// exchange `panels` time-fastest panels of x_tf (panel_stride doubles apart): the ghost rows land in
// ghost[p][n_ghost x ld]
int exchange_plan_run(ctl_handle_s *h, ncclComm_t comm, const ExchangePlan &P, const double *x_tf,
                      size_t panel_stride, int panels, double *ghost);

struct CommState {
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1;
    ExchangePlan mesh;                    // KKT apply, batched Chebyshev, Schur right-hand side
    // ---- device-initiated exchange (halo.cu)
    unsigned long long *d_epoch = nullptr;    // bumped once per sweep replay, after a barrier across ranks
    int *d_err = nullptr;                     // a bounded wait gave up
    int *d_barrier = nullptr;                 // operand of the barrier all-reduce
    long long max_spins = 0;
    std::vector<HaloPlan *> plans;            // live plan instances: their static counters restart with every epoch
};

#define CTL_NCCL(call)                                                                     \
    do {                                                                                   \
        ncclResult_t r__ = (call);                                                         \
        if (r__ != ncclSuccess) {                                                          \
            ctl_set_error(h, std::string(#call) + ": " + ncclGetErrorString(r__));         \
            return CTL_ERR_NCCL;                                                           \
        }                                                                                  \
    } while (0)
