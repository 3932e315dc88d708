// Device side of the aggregation AMG: hierarchy upload and the V-cycle (amg.cu).
#pragma once
#include "amg_setup.h"
#include "sell.cuh"

struct AmgLevelDev {
    int n = 0;                            // rows of this rank (all rows on a replicated level / on one GPU)
    int n_ghost = 0;                      // ghost entries of the level's vector space (distributed levels)
    bool distributed = false;
    double rho = 0.0;
    SellMat A, P, R;
    double *dinv = nullptr;               // n + n_ghost (the ghost part is filled once at setup)
    double *x = nullptr, *b = nullptr;    // owned on levels >= 1 (level 0 uses the caller's)
    double *r = nullptr, *t0 = nullptr, *t1 = nullptr, *t2 = nullptr;   // residual / smoother work vectors
    double *Ainv = nullptr;               // dense inverse on the last level, rows padded to Ainv_ld (even)
    int Ainv_ld = 0;
    HaloPlan *px = nullptr, *pb = nullptr;   // exchanges of the iterates / of the right-hand side (distributed levels)
    HaloPlan *pr = nullptr;               // level 0: exchange of the residual for the restriction (the level-0 space is
                                          // the mesh pattern, shared by every hierarchy; R's columns are not in it)
    HaloPlan *prep = nullptr;             // replicating exchange that delivers this level's right-hand side
};

struct AmgHierarchyDev {
    AmgParams params;
    int nc = 1;                          // components: the levels are the scalar S of I_nc (x) S and every level vector
                                         // holds nc interleaved components per row (set before amg_build; one GPU)
    std::vector<AmgLevelHost> host;      // kept for introspection (ctl_amg_get_csr)
    std::vector<AmgLevelDev> dev;
    std::vector<std::shared_ptr<struct HaloSpace>> spaces;   // multi-GPU: exchange geometry of the levels >= 1 (halo.cu)
    int64_t bytes_per_cycle = 0;         // algorithmic bytes of one V-cycle (byte model, DESIGN.md)
    double *acc_r = nullptr, *acc_z = nullptr, *acc_p = nullptr;   // level-0 work vectors of the accelerated solve
};

// A0 on level 0 may share an existing SELL pattern (fine-level matrices all have the
// mesh pattern); pass nullptr to build one.
int amg_build(ctl_handle_s *h, const HostCSR &A0, const AmgParams &p,
              const std::shared_ptr<SellPattern> &fine_pattern, AmgHierarchyDev &H);
void amg_free(AmgHierarchyDev &H);
// dense_inverse.cu: (A + shift shift^T)^-1 (- shift shift^T when shift is given: the pseudo-inverse of a singular
// symmetric A with normalised kernel vector shift), computed on the device with the host algorithm's arithmetic;
// row-major with row stride *lda_out
int dense_inverse_device(ctl_handle_s *h, const HostCSR &A, const std::vector<double> &shift, double **Ainv_out, int *lda_out);
// upload of an inverse computed on the host (row-major n x n) into the padded device layout
int dense_inverse_upload(ctl_handle_s *h, const std::vector<double> &Ainv, int n, double **Ainv_out, int *lda_out);
// x = `cycles` V-cycles from a zero guess for A x = b (level-0 vectors supplied by the caller).
// Multi-GPU: b_exchanged says that the producer of b has already pushed its boundary rows (level-0 right-hand-side
// plan); the boundary rows of x are pushed by the last kernel of the solve (level-0 iterate plan).
int amg_solve(ctl_handle_s *h, AmgHierarchyDev &H, const double *b, double *x, bool b_exchanged = false);
