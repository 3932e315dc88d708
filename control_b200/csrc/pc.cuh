// In-built block preconditioner state (pc.cu) and its batched kernels (pc_batched.cu).
#pragma once
#include <map>
#include <tuple>

#include "amg.cuh"
#include "common.cuh"
#include "halo_host.cuh"

// pc_batched.cu: one-panel kernels in the time-fastest layout
int pcb_u0_first(ctl_handle_s *h, const double *b0, const double *dinv, double *btil, double *p1, double c);
int pcb_cheb_step(ctl_handle_s *h, const double *dinv, const double *btil, const double *p_prev, const double *p_cur,
                  double *out, double a, double bq, double c);
int pcb_u0_final(ctl_handle_s *h, const double *p, const double *wrap_b, double *u0, double sc, double sc_last);
int pcb_schur_rhs(ctl_handle_s *h, const double *u0, const double *b1, double *out);
int pcb_bc_fixup(ctl_handle_s *h, const int *bc_rows, int n_bc, const double *wrap_b, double *u);
int pcb_panel_to_ts(ctl_handle_s *h, const double *panel_tf, double *ts, size_t stride);
int pcb_ts_to_panel(ctl_handle_s *h, const double *ts, double *panel_tf, size_t stride);

struct PcState {
    ctl_pc_options opts{};
    bool ready = false;
    AmgParams amg;
    int bs = 1;                             // block size the sweeps run with (ctl_set_block_size; 1 when the matrices
                                            // lack the structure I_bs (x) S): S on bs interleaved components

    double *d_mass_dinv = nullptr;          // 1 / diag(assemble(M, bcs))

    std::shared_ptr<SellPattern> fine;      // SELL pattern of the mesh matrix (local rows; of S when bs > 1)
    SellMat Msell;                          // M with constrained rows and columns zeroed
    std::vector<SellMat> off;               // distinct sub/super-diagonal blocks of L_hat
    std::vector<AmgHierarchyDev> hier;      // distinct diagonal blocks of L_hat (+ mass matrix)
    int h_mass = -1;                        // hierarchy of assemble(M, bcs) when Multigrid=True
    std::vector<int> fwd_h, bwd_h;          // hierarchy used at each time step
    std::vector<int> fwd_off, bwd_off;      // off-diagonal matrix used at each time step (-1: none)

    size_t ts_stride = 0;                   // row length of the time-slowest sweep arrays
    double *B = nullptr, *Uf = nullptr, *Ub = nullptr;   // [N][ts_stride]: owned rows, then the ghosts (multi-GPU)
    double *W = nullptr;                    // [ts_stride] right-hand side of the current forward step

    // multi-GPU: device-initiated exchange of the sweep kernels (halo.cuh)
    HaloArena arena;                        // ghost slots and flags of every exchange stream, IPC-shared
    std::shared_ptr<HaloSpace> mesh_space;  // who gathers what through the mesh pattern
    HaloPlan *px0 = nullptr, *pb0 = nullptr;   // level-0 iterates / right-hand sides (shared by all hierarchies)
    cudaGraphExec_t sweep_graph = nullptr;
    int64_t sweep_launches = 0;             // kernels inside one sweep graph
};
