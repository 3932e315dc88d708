/*
 * ctl_b200.h -- C ABI of the B200-native all-at-once KKT solver for `control`.
 *
 * Drop-in boundary for ONE hot path of sleveque/control: the matrix-free KKT operator,
 * the Krylov solve and the in-built block preconditioner of Control.Instationary
 * (SURVEY.md section 8).  Everything is plain C: opaque handle, pointers and sizes, int
 * status codes (0 = ok, < 0 = error; ctl_last_error() gives the message).  No torch /
 * PETSc / Firedrake types cross this boundary.  Each entry point cites the reference
 * interface it replaces (paths relative to the reference checkout).
 *
 * Vector layouts
 *   CTL_LAYOUT_BLOCK_MAJOR  the reference's mixed PETSc vector: 2N contiguous blocks of n
 *                           doubles, [u_0 blocks | u_1 blocks]
 *                           (preconditioner/preconditioner.py:276-287, 658-704).
 *   CTL_LAYOUT_TIME_FASTEST the library's internal layout: two n x ld row-major panels
 *                           (state part, adjoint part), ld = ctl_ld() >= N (power of two,
 *                           N <= 256), padding
 *                           columns are zero.  Used between library calls to avoid the
 *                           two transposes per call.
 * All `double*` vector arguments are DEVICE pointers unless the name ends in `_host`.
 * Matrices are handed over ONCE from host memory (CSR, int32 indices, fp64 values), as
 * assembled by Firedrake/PETSc (`Mat.getValuesCSR()`); the library never renumbers rows.
 */
#ifndef CTL_B200_H
#define CTL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ctl_handle_s *ctl_handle;

enum { CTL_OK = 0, CTL_ERR_ARG = -1, CTL_ERR_CUDA = -2, CTL_ERR_STATE = -3, CTL_ERR_NCCL = -4,
       CTL_ERR_CALLBACK = -5 };

enum { CTL_LAYOUT_BLOCK_MAJOR = 0, CTL_LAYOUT_TIME_FASTEST = 1 };

/* which spatial matrix: mass M (control/control.py:1562), forward operator K = D_v
 * (control/control.py:1887-1896), its adjoint K^T (`adjoint(D_v_i)`, control.py:2905) */
enum { CTL_MAT_M = 0, CTL_MAT_K = 1, CTL_MAT_KT = 2 };

/* Krylov types accepted by solver_parameters["linear_solver"]
 * (preconditioner/preconditioner.py:733) */
enum { CTL_KSP_GMRES = 0, CTL_KSP_FGMRES = 1, CTL_KSP_MINRES = 2 };

/* preconditioner selection for ctl_solve */
enum { CTL_PC_NONE = 0,        /* pc_fn = None: identity (preconditioner.py:342-345)      */
       CTL_PC_BUILTIN = 1,     /* Instationary.construct_pc (control/control.py:1943-2440) */
       CTL_PC_CALLBACK = 2 };  /* user `P=` callable (control/control.py:3245-3258)        */

/* in-built preconditioner structure */
enum { CTL_PCMODE_TRIANGULAR = 0,  /* the reference's block lower-triangular PC            */
       CTL_PCMODE_DIAGONAL = 1 };  /* SPD block-diagonal variant for MINRES (CN only)      */

/* (1,1)-block solver `solver_0` (control/control.py:1953-1991) */
enum { CTL_S0_JACOBI = 0,      /* lambda_v_bounds is None: one Jacobi sweep (1984-1991)    */
       CTL_S0_CHEBYSHEV = 1,   /* Chebyshev/Jacobi with fixed bounds (1967-1982)           */
       CTL_S0_AMG = 2 };       /* Multigrid=True (1954-1965)                               */

/* KSP converged reasons: PETSc's values and sign convention
 * (preconditioner/preconditioner.py:768-770 tests `getConvergedReason() <= 0`) */
enum { CTL_CONVERGED_RTOL = 2, CTL_CONVERGED_ATOL = 3, CTL_CONVERGED_HAPPY_BREAKDOWN = 7,
       CTL_DIVERGED_ITS = -3, CTL_DIVERGED_DTOL = -4, CTL_DIVERGED_BREAKDOWN = -5,
       CTL_DIVERGED_INDEFINITE_PC = -8, CTL_DIVERGED_NANORINF = -9 };

/* Problem description: what Control.Instationary.__init__ / linear_solve fix before the
 * block system is built (control/control.py:1489-1493, 2825-2836). */
typedef struct {
    int32_t n;           /* spatial dofs of space_v (global)                               */
    int32_t n_t;         /* time levels                                                    */
    int32_t CN;          /* 1: trapezoidal/Crank-Nicolson (N = n_t-1), 0: backward Euler   */
    int32_t device;      /* CUDA device ordinal                                            */
    double tau;          /* (T_f - t_0)/(n_t - 1), control/control.py:2831                 */
    double beta;         /* regularisation                                                 */
    double epsilon;      /* BE last-block regularisation, 1e-3 at control/control.py:2836  */
    void *stream;        /* cudaStream_t to launch on; NULL = the library creates one      */
    int32_t rank;        /* row partition: this process' rank ...                          */
    int32_t world;       /* ... of `world` ranks (1 = single GPU)                          */
} ctl_config;

/* Options of the in-built preconditioner: the arguments of
 * Instationary.construct_pc(Multigrid, lambda_v_bounds, ...) (control/control.py:1943)
 * plus the parameters of the aggregation AMG that stands in for
 * `pc_hypre_boomeramg_max_iter: 2` (control/control.py:2060-2067). */
typedef struct {
    int32_t mode;            /* CTL_PCMODE_*                                               */
    int32_t solver_0;        /* CTL_S0_*                                                   */
    double cheb_emin, cheb_emax;   /* lambda_v_bounds                                      */
    int32_t cheb_steps;      /* ksp_max_it of solver_0: 20 (control/control.py:1980)       */
    int32_t amg_cycles;      /* V-cycles per inner solve (default 3; the reference: 2 of hypre) */
    int32_t amg_nu;          /* Chebyshev smoother degree (pre = post) on levels >= 1      */
    int32_t amg_nu_fine;     /* ... on the finest level (0 = amg_nu)                       */
    int32_t amg_max_levels;
    int32_t amg_coarse_max;  /* coarsest level solved with a dense inverse below this size */
    double amg_theta;        /* strength-of-connection threshold                           */
    double amg_lo, amg_hi;   /* smoother interval [lo*rho, hi*rho] of D^-1 A                */
    double amg_acc_lo, amg_acc_hi; /* > 0: Chebyshev-accelerate the V-cycles over this
                                      interval of spec(V-cycle * A); 0 = plain cycles      */
} ctl_pc_options;

/* solver_parameters (preconditioner/preconditioner.py:732-756) */
typedef struct {
    int32_t ksp_type;        /* CTL_KSP_*            ("linear_solver", default fgmres)     */
    int32_t restart;         /* "gmres_restart", PETSc default 30                          */
    int32_t max_it;          /* "maximum_iterations", default 1000                         */
    int32_t pc;              /* CTL_PC_*                                                   */
    double rtol, atol;       /* "relative_tolerance", "absolute_tolerance" (required)      */
    double divtol;           /* "divergence limit", PETSc default 1e4                      */
} ctl_krylov_options;

#define CTL_HISTORY_MAX 1024
typedef struct {
    int32_t its;             /* KSP.getIterationNumber()                                   */
    int32_t reason;          /* KSP.getConvergedReason()                                   */
    int32_t n_mult;          /* operator applications                                      */
    int32_t n_pc;            /* preconditioner applications                                */
    double rnorm;            /* last monitored residual norm                               */
    double ref_norm;         /* norm the relative tolerance refers to                      */
    int32_t n_history;
    double history[CTL_HISTORY_MAX];   /* what the KSP monitor would print (it = 0 first)  */
    double seconds_total, seconds_mult, seconds_pc;   /* device time (CUDA events)         */
} ctl_solve_result;

/* user preconditioner, the `P=` hook: pc_fn(u_0, u_1, b_0, b_1)
 * (control/control.py:3245-3258; called from Preconditioner.apply,
 * preconditioner/preconditioner.py:620-627).  b and u are DEVICE pointers to block-major
 * vectors of 2*N*n doubles; b is already BC-projected, u is zero on entry.  Return 0. */
typedef int (*ctl_pc_callback)(void *user, const double *b, double *u);

/* ---- lifetime: MultiBlockSystem.__init__ / `del system` (preconditioner.py:217-335,
 *      control/control.py:3323-3326) */
int ctl_create(const ctl_config *cfg, ctl_handle *out);
/* world > 1: collective once ctl_pc_setup has run (the preconditioner's exchange arena is released behind two
 * barriers across the ranks): every rank destroys its handle at the same point of its call sequence */
int ctl_destroy(ctl_handle h);
const char *ctl_last_error(ctl_handle h);     /* h may be NULL: error of a failed create  */
const char *ctl_version(void);

/* ---- matrices: replace the 8N-4 (CN) / 6N-4 (BE) `assemble(block_ij)` calls of
 *      MultiBlockSystem.__init__ (preconditioner/preconditioner.py:305-328) by the two or
 *      three distinct spatial matrices they are built from (control/control.py:2889-2978).
 *      One shared pattern; `level` = time level of K / K^T, or -1 = the same at all levels. */
int ctl_set_pattern(ctl_handle h, const int32_t *indptr_host, const int32_t *indices_host,
                    int64_t nnz);
int ctl_set_values(ctl_handle h, int which, int level, const double *values_host);
/* homogeneous Dirichlet dofs: DirichletBCNullspace(bcs_v)
 * (preconditioner/preconditioner.py:158-197; control/control.py:2851-2862) */
int ctl_set_bc(ctl_handle h, const int32_t *dofs_host, int32_t count);
/* block size of a vector-valued space: PETSc's Mat block size with interleaved numbering, dof = bs node + comp
 * (Firedrake's VectorFunctionSpace).  bs = 1 (the default) is the scalar path.  With bs > 1, ctl_pc_setup checks
 * whether EVERY matrix of the time sweeps -- M, each distinct diagonal block and its AMG hierarchy, the
 * Multigrid=True mass hierarchy, each off-diagonal block -- is I_bs (x) S: no entry couples two components and the
 * bs component blocks are bitwise equal (absent entries and stored zeros count as 0; a Dirichlet list that is not
 * node-closed breaks it).  If so, the sweeps are set up and run on the scalar S, each product acting on bs
 * interleaved components (every AMG hierarchy is that of S with coarse_max replaced by ceil(coarse_max / bs));
 * otherwise the handle takes the bs = 1 path.  The KKT apply and the batched parts of the preconditioner do not
 * change.  CTL_ERR_ARG unless bs is 1, 2 or 3 and divides n, and for bs > 1 with world > 1 (block-scalar sweeps
 * run on one GPU).  Drops a preconditioner that is already set up (call ctl_pc_setup again). */
int ctl_set_block_size(ctl_handle h, int32_t bs);
/* finish setup (uploads, eliminations); must precede apply/solve.  Drops a set-up preconditioner: with world > 1
 * that release is collective like ctl_destroy, so every rank assembles at the same point */
int ctl_assemble(ctl_handle h);

/* ---- sizes */
int32_t ctl_n_blocks(ctl_handle h);            /* N: n_t-1 (CN) or n_t (BE)                */
int32_t ctl_ld(ctl_handle h);                  /* padded row length of the internal layout */
int32_t ctl_n_local(ctl_handle h);             /* rows owned by this rank                  */
int32_t ctl_row_begin(ctl_handle h);           /* first owned global row                   */
int64_t ctl_vec_len(ctl_handle h, int layout); /* doubles per (local) vector               */
int ctl_convert_layout(ctl_handle h, const double *src, int src_layout, double *dst,
                       int dst_layout);

/* ---- y = A x : MultiBlockSystemMatrix.mult (preconditioner/preconditioner.py:375-543),
 *      the callback PETSc invokes through Mat().createPython (720-722). */
int ctl_kkt_apply(ctl_handle h, const double *x, double *y, int layout);

/* ---- in-built preconditioner: Instationary.construct_pc (control/control.py:1943-2440)
 *      wrapped as Preconditioner.apply (preconditioner/preconditioner.py:562-656). */
int ctl_pc_default_options(ctl_pc_options *opts);
int ctl_pc_setup(ctl_handle h, const ctl_pc_options *opts);
/* block size the preconditioner that is set up runs its sweeps with (1 when the matrices lack the structure
 * ctl_set_block_size asks for); -1 before ctl_pc_setup */
int32_t ctl_pc_block_size(ctl_handle h);
int ctl_pc_apply(ctl_handle h, const double *b, double *u, int layout);
/* the raw pc_fn(u_0, u_1, b_0, b_1) without the nullspace wrapping (what a user would
 * pass back through `P=`) */
int ctl_pc_fn(ctl_handle h, const double *b, double *u, int layout);
int ctl_set_pc_callback(ctl_handle h, ctl_pc_callback fn, void *user);

/* ---- KSP solve: MultiBlockSystem.solve (preconditioner/preconditioner.py:337-786).
 *      u: initial guess in, solution out.  Non-convergence is reported through
 *      result->reason, never as an error code (the Python layer raises the reference's
 *      RuntimeError("Solver failed to converge")). */
int ctl_krylov_default_options(ctl_krylov_options *opts);
int ctl_solve(ctl_handle h, const double *b, double *u, int layout,
              const ctl_krylov_options *opts, ctl_solve_result *result);
/* same, host buffers (block-major), copies inside: the end-to-end call */
int ctl_solve_host(ctl_handle h, const double *b_host, double *u_host,
                   const ctl_krylov_options *opts, ctl_solve_result *result);

/* ---- diagnostics on device vectors */
/* ||b - A x||_2 with the projected operator (SURVEY.md section 8c) */
int ctl_kkt_residual_norm(ctl_handle h, const double *b, const double *x, int layout,
                          double *out);
/* residual of the outer Picard / Gauss-Newton loop (replaces non_linear_res_eval, control/control.py:2442-2818)
 * on DEVICE vectors: r = b - A x with the rows of constrained dofs zeroed, where b is the right-hand side of
 * linear_solve for the problem data and A carries D_v at the iterate x (ctl_set_values per level first).  r is
 * the residual AFTER the T_1 / T_2 transforms, i.e. the right-hand side of the increment solve; *norm_host is
 * || T^-1 r ||_2, the norm of the reference's (untransformed) residual, reduced over all ranks. */
int ctl_nonlinear_residual(ctl_handle h, const double *b, const double *x, double *r, int layout,
                           double *norm_host);
/* discrete objective J_h (SURVEY.md section 8c); v, zeta, v_hat: n_t levels x n, host */
int ctl_objective_host(ctl_handle h, const double *v_host, const double *zeta_host,
                       const double *v_hat_host, double *out);
/* the same on DEVICE arrays (n_t levels x n_local, level-major: this rank's rows); the scalar is returned to the
 * host.  Several ranks: ghost entries are fetched from their owners, the sums are all-reduced, every rank
 * receives J_h. */
int ctl_objective(ctl_handle h, const double *v, const double *zeta, const double *v_hat,
                  double *out_host);
/* ---- right-hand sides of linear_solve from NODAL data (control/control.py:2980-3243) for homogeneous
 *      Dirichlet data; inhomogeneous data are added afterwards with ctl_lift_bc.  v_hat, f_nodal are DEVICE arrays
 *      of n_t levels x n (the reference's
 *      cofunctions are M v_hat_i, M f_i for interpolated data); v_0_host: the initial condition
 *      (n doubles, host: ALL n entries on every rank) or NULL = 0; b: DEVICE block-major output (this rank's
 *      rows), T_1 / T_2 applied.  Several ranks: v_hat, f_nodal hold this rank's rows (n_t x n_local); the ghost
 *      entries the products gather are fetched from their owners. */
int ctl_build_rhs(ctl_handle h, const double *v_hat, const double *f_nodal, const double *v_0_host,
                  double *b);
/* ---- lifting of inhomogeneous, time-dependent Dirichlet data of the state (the reference's `v_inhom`,
 *      control/control.py:2993-3124 BE, 3137-3212 CN): b <- b - T(L(g)) on the unconstrained rows, where L(g) is what
 *      the boundary values contribute through the constrained COLUMNS of M and K to the rows of linear_solve
 *      (BE: L_0[i] = tau M g_i for i < n_t-1, L_1[i] = tau K_i g_i + M g_i - M g_{i-1}; CN: L_0[i] = h M (g_{i+1} + g_i),
 *      L_1[i] = (h K_{i+1} + M) g_{i+1} + (h K_i - M) g_i, the g_0 terms dropped, h = tau/2) and T = (T_1, T_2) for
 *      CN, the identity for BE.  Constrained rows of b are not touched.  The lifting is additive, so it composes with
 *      ctl_build_rhs, a host-built b, and the b handed to ctl_nonlinear_residual (with K_i at the iterate: after new
 *      ctl_set_values + ctl_assemble the next call uses the new values).
 *      g: DEVICE, n_t levels x n_bc (level-major), columns in the order of the ctl_set_bc list; every rank passes all
 *         n_t x n_bc values (no communication).
 *      b: DEVICE, in and out, this rank's rows in `layout`.
 *      Errors: CTL_ERR_STATE before ctl_assemble; CTL_ERR_ARG for an unknown layout, or a NULL g / b when the handle
 *      has Dirichlet dofs.  With no Dirichlet dofs the call does nothing.  Asynchronous on the handle's stream. */
int ctl_lift_bc(ctl_handle h, const double *g, double *b, int layout);

/* ---- AMG introspection (tests compare the hierarchy with the oracle's).  A block hierarchy (ctl_pc_block_size > 1)
 *      is that of the scalar S: level sizes, matrices and aggregates describe the scalar levels; ctl_amg_solve takes
 *      n-vectors in the interleaved layout (16-byte aligned for bs = 2) and solves every component; ctl_time_amg counts
 *      the matrix bytes once and the vector bytes bs times (the Jacobi diagonal, one entry per node, once). */
int32_t ctl_amg_num_hierarchies(ctl_handle h);
int32_t ctl_amg_num_levels(ctl_handle h, int32_t hierarchy);
int ctl_amg_level_size(ctl_handle h, int32_t hierarchy, int32_t level, int32_t *n,
                       int64_t *nnz_A, int64_t *nnz_P);
/* copy level matrices out (host CSR); which: 0 = A, 1 = P */
int ctl_amg_get_csr(ctl_handle h, int32_t hierarchy, int32_t level, int which,
                    int32_t *indptr_host, int32_t *indices_host, double *values_host);
int ctl_amg_get_aggregates(ctl_handle h, int32_t hierarchy, int32_t level, int32_t *agg_host);
/* x = AMG(b): `cycles` V-cycles from a zero guess on hierarchy `hierarchy`; device n-vectors */
int ctl_amg_solve(ctl_handle h, int32_t hierarchy, const double *b, double *x);

/* ==== Instationary Stokes control: Control.Instationary.incompressible_linear_solve
 *      (control/control.py:3592-4725).  The outer system couples the heat-type KKT system of
 *      the velocity space (block_00, control.py:3750-3957) with the divergence blocks
 *      tau B^T / tau B (block_01 / block_10, 3755-3766) under sub-block T transforms
 *      (preconditioner/preconditioner.py:471-525) and ConstantNullspace on the pressure blocks
 *      (preconditioner.py:133-155).  It is described by TWO handles -- `velocity` (M_v, K_v,
 *      velocity Dirichlet dofs) and `pressure` (M_p, K_p, no bcs), same n_t / tau / beta / CN /
 *      device / stream -- plus the divergence matrix B (n_p x n_v CSR, host).  Vectors are
 *      DEVICE pointers, block-major: [2N blocks of n_v (v | zeta) | 2N blocks of n_p (mu | p)].
 *      Errors are reported through ctl_last_error(velocity).
 *      Several GPUs (one process each): both handles carry the same rank / world > 1 and have been through
 *      ctl_comm_init.  Every rank passes the GLOBAL B; velocity and pressure rows are each split by PETSc's rule
 *      (the handles' own partitions), and every entry point works on this rank's rows: the outer vector is
 *      [2N blocks of n_v_local | 2N blocks of n_p_local] and ctl_stokes_vec_len is that local length.  The
 *      divergence products exchange the rows of the other space they read through NCCL; the pressure means, the
 *      Krylov dots and the residual norm are summed over all ranks, so every rank receives the same global values.
 *      All calls are collective.  Block-scalar velocity sweeps (ctl_set_block_size > 1) stay on one GPU. */
typedef struct ctl_stokes_s *ctl_stokes;

/* the in-built pressure-Schur preconditioner (control/control.py:4299-4687) */
typedef struct {
    ctl_pc_options velocity;   /* construct_pc of the inner heat-type solve (4346-4353)             */
    int32_t inner_its;         /* GMRES iterations of the block_00 solve: 5 (4355-4361)             */
    int32_t mass_p;            /* solver_M_p: CTL_S0_CHEBYSHEV (lambda_p_bounds) or CTL_S0_JACOBI   */
    int32_t mass_p_steps;      /* 20 (4311-4333)                                                    */
    double lambda_p_min, lambda_p_max;
    /* solver_K_p: ONE cycle of the aggregation AMG on the Neumann Laplacian K_p, coarsest level
     * smoothed only (stands in for hypre BoomerAMG x1, control/control.py:4300-4309) */
    int32_t amg_p_nu, amg_p_max_levels, amg_p_coarse_max, amg_p_cycles;
    double amg_p_theta, amg_p_lo, amg_p_hi;
} ctl_stokes_pc_options;

/* CTL_ERR_ARG: the handles differ in n_t, CN, tau, beta, rank, world, device or stream, the pressure handle has
 * Dirichlet dofs, or B has a column out of range; CTL_ERR_STATE: a handle is not assembled, or (world > 1) has not
 * been through ctl_comm_init */
int ctl_stokes_create(ctl_handle velocity, ctl_handle pressure, const int32_t *B_indptr_host,
                      const int32_t *B_indices_host, const double *B_values_host, ctl_stokes *out);
int ctl_stokes_destroy(ctl_stokes s);
int64_t ctl_stokes_vec_len(ctl_stokes s);      /* 2 N (n_v_local + n_p_local); n_v + n_p on one GPU */
/* y = A x: MultiBlockSystemMatrix.mult with sub_n_blocks = 2 (preconditioner.py:375-543) */
int ctl_stokes_apply(ctl_stokes s, const double *x, double *y);
int ctl_stokes_pc_default_options(ctl_stokes_pc_options *opts);
/* Values (HOST, on the pressure handle's pattern) of the Laplacian `K_p = inner(grad(p_trial), grad(p_test)) dx`
 * that solver_K_p inverts (control/control.py:3746, 4300-4309).  Without this call the forward matrix of the
 * pressure handle is used, which is the same matrix for the Stokes forward operator.  Needed when the forward
 * form restricted to the pressure space (block_10_int_p = tau D_p_i + M_p, control/control.py:3787-3789) is NOT
 * the Laplacian: Navier-Stokes Picard iterations (per-level convection-diffusion D_p_i), forward forms with a
 * reaction term.  NULL restores the default.  Call before ctl_stokes_pc_setup. */
int ctl_stokes_set_laplacian_p(ctl_stokes s, const double *values_host);
int ctl_stokes_pc_setup(ctl_stokes s, const ctl_stokes_pc_options *opts);
/* Preconditioner.apply around pc_fn (with the nullspace wrapping) / the raw pc_fn */
int ctl_stokes_pc_apply(ctl_stokes s, const double *b, double *u);
int ctl_stokes_pc_fn(ctl_stokes s, const double *b, double *u);
/* user preconditioner of the outer Stokes system: the `P=` argument of incompressible_linear_solve
 * (control/control.py:3592-3594, 4686-4689).  fn(user, b, u) receives DEVICE vectors of ctl_stokes_vec_len doubles
 * in the outer block-major layout, b projected (Dirichlet rows of the velocity blocks zero, pressure blocks mean
 * free), u zero, and fills u; a non-zero return aborts the solve (flag_errors, preconditioner.py:64-72).  Selected
 * with opts->pc = CTL_PC_CALLBACK. */
int ctl_stokes_set_pc_callback(ctl_stokes s, ctl_pc_callback fn, void *user);
/* MultiBlockSystem.solve of the outer system (control/control.py:4273-4297, 4688-4693);
 * opts->pc: CTL_PC_NONE or CTL_PC_BUILTIN */
int ctl_stokes_solve(ctl_stokes s, const double *b, double *u, const ctl_krylov_options *opts,
                     ctl_solve_result *result);
/* lifting of inhomogeneous velocity Dirichlet data into an outer right-hand side b (DEVICE, block-major, in and out):
 * the velocity rows as ctl_lift_bc on the velocity handle, and the divergence rows b_1_0[i] -= tau B g_{i+1} (CN) /
 * tau B g_i (BE), then T_2 for CN (control/control.py:4107-4119, 4207-4219), with the constrained columns of B as
 * handed to ctl_stokes_create.  g: DEVICE, n_t x n_bc of the velocity handle, level-major.  Error codes as
 * ctl_lift_bc, reported through ctl_last_error(velocity). */
int ctl_stokes_lift_bc(ctl_stokes s, const double *g, double *b);
/* Residual of the Navier-Stokes Picard loop (res_eval of incompressible_non_linear_solve, control/control.py:
 * 4979-5072) on DEVICE vectors of ctl_stokes_vec_len doubles, outer block-major layout: r = b - A_raw x, with A_raw
 * the fused KKT operator on the velocity blocks (the K values the velocity handle holds: D_v at the iterate, after
 * ctl_set_values / ctl_assemble), plus tau T(B^T x_p) on the velocity rows and tau T(B x_v) on the pressure rows,
 * WITHOUT the ConstantNullspace corrections of ctl_stokes_apply -- the reference's residual uses raw products.
 * Constrained velocity rows of r are zero; D_p does not enter.  *norm_host = sqrt(||T^-1 r_v||^2 +
 * ||T^-1 r_p||^2 / tau^2), the norm of the untransformed, unscaled parts (r00, r01, r10, r11) the loop tests (T_1 on
 * the first N velocity blocks and the last N pressure blocks, T_2 on the others; identity for BE).  b and x are not
 * modified; r must not alias them.  CTL_ERR_ARG for null or aliased pointers, CTL_ERR_STATE if a handle is not
 * assembled; messages through ctl_last_error(velocity). */
int ctl_stokes_nonlinear_residual(ctl_stokes s, const double *b, const double *x, double *r, double *norm_host);
/* time `reps` back-to-back launches of the batched divergence products on one time panel (CUDA
 * events on the stream; the panels exceed L2 at config C4).  out[0] = tau B X, average ms;
 * out[1] = its algorithmic bytes (12 nnz_B + 4 (n_p + 1) + 8 N (n_v + n_p)); out[2] = Y += tau B^T X,
 * ms; out[3] = its bytes (the same + 8 N n_v for the accumulate) */
int ctl_stokes_time(ctl_stokes s, int reps, double *out4_host);

/* ---- host-only probe of the AMG setup (no GPU needed; the CPU test-suite compares it with the oracle):
 *      sets up the hierarchy of the n x n CSR matrix with the AMG options of `opts` (NULL = defaults) and
 *      reports up to 16 levels: rows, entries above 1e-13 x the largest one, spectral bound rho, and the
 *      aggregate id of every fine row */
int ctl_amg_setup_probe(const int32_t *indptr_host, const int32_t *indices_host, const double *values_host,
                        int32_t n, const ctl_pc_options *opts, int32_t *n_levels, int32_t *level_n16,
                        int64_t *level_nnz16, double *level_rho16, int32_t *aggregates_n);

/* ---- multi-GPU (one process per GPU): the 128-byte ncclUniqueId is created on rank 0
 *      with ctl_comm_unique_id and distributed by the caller (torch.distributed).  With world > 1 every call that
 *      communicates is collective -- the entry points that apply, precondition or solve, ctl_pc_setup,
 *      ctl_stokes_create / _pc_setup, and the releases of ctl_destroy, ctl_assemble, ctl_set_block_size and
 *      ctl_stokes_destroy: all ranks make them in the same order */
int ctl_comm_unique_id(void *id128_host);
int ctl_comm_init(ctl_handle h, const void *id128_host);

/* ---- instrumentation */
int64_t ctl_kernel_launches(ctl_handle h);     /* kernels launched by this handle so far   */
/* time `reps` back-to-back launches of the fused KKT-apply kernel alone (time-fastest
 * layout, CUDA events on the handle's stream); average milliseconds per launch */
int ctl_time_kkt_apply(ctl_handle h, const double *x_tf, double *y_tf, int reps, float *ms);

/* time the kernels of the time sweeps in isolation on AMG hierarchy `hierarchy` (CUDA
 * events on the handle's stream around `reps` launches).  flush_l2 != 0: cold operands --
 * every launch of the two fine-level kernels works on its own set of vectors and the sets
 * rotate through more than twice the L2 capacity (inputs larger than L2); the inner solve
 * is preceded by the overwrite of a 256 MB buffer, whose time is subtracted.  out[0] = level-0 smoother step, ms; out[1] = its algorithmic
 * bytes; out[2] = level-0 residual SpMV, ms; out[3] = its bytes; out[4] = one inner solve
 * (all cycles, all levels), ms; out[5] = its algorithmic bytes; out[6] = kernels per solve */
int ctl_time_amg(ctl_handle h, int32_t hierarchy, int reps, int flush_l2, double *out7);

#ifdef __cplusplus
}
#endif
#endif /* CTL_B200_H */
