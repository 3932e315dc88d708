// Host-side smoothed-aggregation setup (amg_setup.cpp).  Step-for-step the algorithm of
// oracle/amg.py; see that file's header for the definition and DESIGN.md for why this
// replaces hypre BoomerAMG (control/control.py:2056-2067).
#pragma once
#include <vector>

#include "common.cuh"

enum { AMG_COARSE_INVERSE = 0,          // dense inverse
       AMG_COARSE_PINV_CONSTANT = 1,    // pseudo-inverse, kernel = image of the constants (Neumann Laplacian)
       AMG_COARSE_SMOOTH = 2 };         // smoother only

struct AmgParams {
    double theta = 0.08;
    double theta_decay = 0.5;   // strength threshold on level l: theta * theta_decay^l
    int max_levels = 10;
    int coarse_max = 2500;  // dense inverse below this size: ONE 2205^2 GEMV (39 MB, L2-resident) at C2 instead of two
                            // more levels of ~10 dependent launches each (round 2; was 600)
    int nu = 3;          // smoother degree on levels >= 1
    int nu_fine = 0;     // smoother degree on level 0 (0 = nu)
    double lo = 0.25, hi = 1.0;
    int cycles = 3;      // see oracle/amg.py::solve for why not the reference's 2
    double acc_lo = 0.0, acc_hi = 1.0;   // > 0: Chebyshev-accelerated cycles (oracle/amg.py::solve)
    int coarse = 0;                      // AMG_COARSE_*: what happens on the coarsest level
    int device_inverse = 1;              // 1: the dense inverse of the coarsest level is left to the device
                                         // (dense_inverse.cu: 2205 rows at C2 = 5 s on one host core, 50 ms on the GPU);
                                         // 0: computed here (host-only checks)
};

struct AmgLevelHost {
    HostCSR A;                 // level operator
    std::vector<double> dinv;  // 1 / diag(A)
    double rho = 0.0;          // Gershgorin bound of D^-1 A
    std::vector<int> agg;      // aggregate id per row (-1 = not aggregated); empty on the last level
    HostCSR P, R;              // prolongation (n x n_coarse) and R = P^T; empty on the last level
    std::vector<double> Ainv;  // dense inverse, row-major (last level, n <= 4096); empty when left to the device:
    int coarse_inverse = 0;    // ... then AMG_COARSE_INVERSE + 1 / AMG_COARSE_PINV_CONSTANT + 1 says what to compute,
    std::vector<double> coarse_shift;   // and this is the normalised kernel vector of the pseudo-inverse
    bool has_inverse() const { return !Ainv.empty() || coarse_inverse != 0; }
};

// host threads of the preconditioner set-up: the environment variable CTL_SETUP_THREADS when it is set (a limit for
// shared hosts), `fallback` otherwise
int setup_threads(int fallback);

// A must have sorted column indices.  Returns the levels, finest first.
// threads: host threads for the row-parallel phases (0 = all hardware threads, up to 32, or setup_threads); the
// result does not depend on it
void amg_setup_host(const HostCSR &A, const AmgParams &p, std::vector<AmgLevelHost> &levels, int threads = 0);

// helpers shared with tests / other units
void csr_transpose(const HostCSR &A, HostCSR &At);
void csr_matmat(const HostCSR &A, const HostCSR &B, HostCSR &C, int threads = 1);
