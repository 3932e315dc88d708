"""Host-side mirror of ``Control.Stationary`` for the heat-type path (SURVEY.md section 8f rank 4:
"Stationary problems as the N = 1 case"; control/control.py:100-800).

The stationary KKT system [[M, D_v^T], [D_v, -M/beta]] (control/control.py:549-560) and its block
preconditioner (351-450) ARE the trapezoidal system and preconditioner of the instationary path with one
time block: with n_t = 2, tau = 2 and the forward matrix K' = D_v - M the block tables
(control/control.py:2929-2958) give

    block_00 = (tau/2) M = M          block_01 = (tau/2) K'^T + M = D_v^T
    block_10 = (tau/2) K' + M = D_v   block_11 = -(tau/2)/beta M = -M/beta

T_1 = T_2 = I for a single block, the (1,1) solve is ``(2/tau) M~^-1``, and both Schur solves use
``(tau/2) K' + M + (tau/2)/sqrt(beta) M = D_v + M/sqrt(beta)`` (transposed in the second one) -- exactly
``solver_1`` / ``solver_2`` of 395-417.  So the stationary drivers run on the same device handle, kernels and
Krylov code as the instationary ones; nothing here computes on the host beyond the small vector algebra the
reference does in Firedrake (right-hand sides, lifting, residuals of the non-linear loop).
"""
import numpy as np
import scipy.sparse as sp

from .outer_loop import picard
from .system import MultiBlockSystem, fgmres_defaults, gmres_defaults

__all__ = ["Stationary"]


class Stationary:
    def __init__(self, M, forward_matrix, *, desired_state=None, force_f=None, force_function=None, beta=1.0e-3,
                 Gauss_Newton=False, bc_dofs=(), bc_values=None, device=None):
        """``M``: mass matrix (scipy CSR).  ``forward_matrix``: the matrix of ``forward_form`` on M's pattern,
        or a callable ``(v, gauss_newton) -> CSR`` returning ``construct_D_v`` (control/control.py:314-324) at
        the state ``v``.  ``desired_state()`` -> (M @ v_hat, v_hat) and ``force_f()`` -> M @ f, the assembled
        values of the reference's callables (control/control.py:118-134).  ``bc_values``: None (homogeneous) or
        the values of the state at ``bc_dofs``."""
        if force_f is not None and force_function is not None:
            raise TypeError("give either force_f or force_function")
        self._M = M.tocsr()
        self._forward_matrix = forward_matrix
        self._desired_state = desired_state
        self._force = force_f if force_f is not None else force_function
        self._beta = float(beta)
        self._Gauss_Newton = bool(Gauss_Newton)
        self._bc_dofs = np.ascontiguousarray(bc_dofs, dtype=np.int32)
        self._bc_values = None if bc_values is None else np.asarray(bc_values, dtype=float)
        self._n = self._M.shape[0]
        self._v = np.zeros(self._n)
        self._zeta = np.zeros(self._n)
        self._true_v = None
        self._system = None
        self._device = device
        self.last_ksp = None
        self.non_linear_history = []

    # ------------------------------------------------------------------ helpers
    def construct_D_v(self, v_old):                      # control/control.py:314-324
        if callable(self._forward_matrix):
            return self._forward_matrix(v_old, self._Gauss_Newton)
        return self._forward_matrix

    def _assembled_force(self):
        return np.zeros(self._n) if self._force is None else np.asarray(self._force(), dtype=float)

    def _assembled_desired_state(self):
        if self._desired_state is None:
            self._true_v = np.zeros(self._n)
            return np.zeros(self._n)
        v_d, self._true_v = self._desired_state()
        return np.asarray(v_d, dtype=float)

    def _bc(self, b):
        b[..., self._bc_dofs] = 0.0

    def _shifted(self, D_v):
        """K' = D_v - M on the shared pattern (structural zeros kept)."""
        D_v = D_v.tocsr()
        if not D_v.has_sorted_indices:
            D_v = D_v.sorted_indices()
        M = self._M if self._M.has_sorted_indices else self._M.sorted_indices()
        if D_v.nnz != M.nnz or not (np.array_equal(D_v.indptr, M.indptr) and np.array_equal(D_v.indices, M.indices)):
            raise ValueError("M and the forward matrix must share one sparsity pattern (keep structural zeros)")
        return sp.csr_matrix((D_v.data - M.data, M.indices, M.indptr), shape=M.shape)

    def _ensure_system(self, D_v):
        K = self._shifted(D_v)
        if self._system is None:
            self._system = MultiBlockSystem(self._M, K, n_t=2, beta=self._beta, CN=True, time_interval=(0.0, 2.0),
                                            bc_dofs=self._bc_dofs, device=self._device)
        else:
            self._system.set_K(K)
        return self._system

    def close(self):
        if self._system is not None:
            self._system.close()
            self._system = None
        if getattr(self, "_stokes", None) is not None:
            self._stokes.close()
            self._stokes = None

    def print_error(self):                              # control/control.py:303-312
        if self._true_v is None:
            return None
        d = self._v - self._true_v
        error = float(np.sqrt(abs(d @ (self._M @ d))))
        print(f"Estimated error in the L2-norm: {error:.16e}")
        return error

    # ------------------------------------------------------------------ linear_solve
    def linear_solve(self, *, P=None, solver_parameters=None, Multigrid=False, lambda_v_bounds=None, v_d=None, f=None,
                     print_error=True, create_output=False, plots=False, **amg):
        """control/control.py:489-628.  ``v_d`` / ``f``: ready right-hand sides (used as they are), or None
        for the assembled desired state / force, lifted when the Dirichlet data are inhomogeneous."""
        n, M = self._n, self._M
        D_v = self.construct_D_v(self._v)
        v_inhom = None
        if self._bc_values is not None:                 # 520-526
            v_inhom = np.zeros(n)
            v_inhom[self._bc_dofs] = self._bc_values
        if f is None:                                   # construct_f, 326-336
            b_1 = self._assembled_force()
            if v_inhom is not None:
                b_1 = b_1 - D_v @ v_inhom
                self._bc(b_1)
        else:
            b_1 = np.array(f, dtype=float)
        if v_d is None:                                 # construct_v_d, 338-349
            b_0 = self._assembled_desired_state()
            if v_inhom is not None:
                b_0 = b_0 - M @ v_inhom
                self._bc(b_0)
        else:
            b_0 = np.array(v_d, dtype=float)
        if solver_parameters is None:                   # 562-568
            solver_parameters = gmres_defaults(print_error)
        system = self._ensure_system(D_v)
        if P is None:                                   # 541-545
            system.setup_preconditioner(lambda_v_bounds=lambda_v_bounds, Multigrid=Multigrid, **amg)
            pc_fn = "builtin"
        else:
            pc_fn = P
        v = np.zeros((1, n))
        zeta = np.zeros((1, n))
        self.last_ksp = system.solve(v, zeta, b_0[None].copy(), b_1[None].copy(), solver_parameters=solver_parameters,
                                     pc_fn=pc_fn)
        v, zeta = v[0], zeta[0]
        if v_inhom is not None:                         # 586-589
            v = v + v_inhom
        # set_v / set_zeta re-apply the boundary conditions (264-283)
        v[self._bc_dofs] = 0.0 if self._bc_values is None else self._bc_values
        self._bc(zeta)
        self._v, self._zeta = v, zeta
        if print_error:
            self.print_error()
        return self.last_ksp

    # ------------------------------------------------------------------ Stokes / Navier-Stokes control
    def set_space_p(self, space_p):
        """``space_p``: dict with the divergence matrix ``B`` (n_p x n_v), the pressure mass matrix ``M_p``, the
        pressure Laplacian ``K_p`` and ``forward_matrix_p``: the forward form on the pressure space -- a CSR
        matrix on M_p's pattern or a callable ``(v, gauss_newton) -> CSR`` (``block_10_p``,
        control/control.py:971); default ``K_p`` (the Stokes forward operator)."""
        self._space_p = space_p

    def _D_p(self, space_p, v_old):
        fp = space_p.get("forward_matrix_p")
        if fp is None:
            return space_p["K_p"]
        return fp(v_old, self._Gauss_Newton) if callable(fp) else fp

    def incompressible_linear_solve(self, nullspace_p=None, *, space_p=None, P=None, solver_parameters=None,
                                    Multigrid=False, lambda_v_bounds=None, lambda_p_bounds=None, v_d=None, f=None,
                                    div_v=None, div_zeta=None, print_error=True, create_output=False, plots=False,
                                    amg=None, amg_p=None):
        """control/control.py:802-1201.  The outer system [[KKT_v, B^T], [B, 0]] runs on the instationary Stokes
        handle with one time block (n_t = 2, tau = 2, forward matrices shifted by the mass matrices, see the module
        header): that system couples with ``tau B`` = 2 B, so the divergence rows are handed over scaled by 2 and
        the pressures come back scaled by 1/2 -- a diagonal scaling of the unknowns under which the in-built
        preconditioner (986-1084 = control/control.py:4337-4513 with one block) is consistent."""
        from .stokes import StokesSystem
        if space_p is None:
            space_p = getattr(self, "_space_p", None)
            if space_p is None:
                raise ValueError("Undefined space_p")                   # 815-819
        else:
            self.set_space_p(space_p)
        if nullspace_p not in (None, "constant"):
            raise ValueError("only the constant pressure nullspace is supported")
        if P is not None:
            raise NotImplementedError("user preconditioners are not wired for the Stokes system")
        n, M, B = self._n, self._M, space_p["B"]
        M_p = space_p["M_p"].tocsr()
        n_p = M_p.shape[0]
        D_v = self.construct_D_v(self._v)
        D_p = self._D_p(space_p, self._v).tocsr()
        v_inhom = None
        if self._bc_values is not None:
            v_inhom = np.zeros(n)
            v_inhom[self._bc_dofs] = self._bc_values
        if f is None:                                   # construct_f, 326-336
            b_01 = self._assembled_force()
            if v_inhom is not None:
                b_01 = b_01 - D_v @ v_inhom
                self._bc(b_01)
        else:
            b_01 = np.array(f, dtype=float)
        if v_d is None:                                 # construct_v_d, 338-349
            b_00 = self._assembled_desired_state()
            if v_inhom is not None:
                b_00 = b_00 - M @ v_inhom
                self._bc(b_00)
        else:
            b_00 = np.array(v_d, dtype=float)
        if div_v is None:                               # 866-873
            b_10 = np.zeros(n_p) if v_inhom is None else -(B @ v_inhom)
        else:
            b_10 = np.array(div_v, dtype=float)
        b_11 = np.zeros(n_p) if div_zeta is None else np.array(div_zeta, dtype=float)
        if solver_parameters is None:                   # 1088-1094
            solver_parameters = fgmres_defaults(print_error, max_it=50)
        K_shift = self._shifted(D_v)
        D_p_shift = sp.csr_matrix((D_p.data - M_p.data, M_p.indices, M_p.indptr), shape=M_p.shape)
        if getattr(self, "_stokes", None) is None:
            self._stokes = StokesSystem(M, K_shift, B, M_p, space_p["K_p"], n_t=2, beta=self._beta, CN=True,
                                        time_interval=(0.0, 2.0), bc_dofs_v=self._bc_dofs, device=self._device,
                                        D_p=D_p_shift)
        else:
            self._stokes.set_forward(K_shift, D_p_shift)
        system = self._stokes
        system.setup_preconditioner(lambda_v_bounds=lambda_v_bounds, lambda_p_bounds=lambda_p_bounds, amg=amg,
                                    amg_p=amg_p, Multigrid=Multigrid)
        u_0 = np.zeros((2, n))
        u_1 = np.zeros((2, n_p))
        self.last_ksp = system.solve(u_0, u_1, np.stack([b_00, b_01]), 2.0 * np.stack([b_10, b_11]),
                                     solver_parameters=solver_parameters, pc_fn="builtin")
        v, zeta = u_0[0].copy(), u_0[1].copy()
        if v_inhom is not None:                         # 1107-1110
            v = v + v_inhom
        v[self._bc_dofs] = 0.0 if self._bc_values is None else self._bc_values
        self._bc(zeta)
        self._v, self._zeta = v, zeta
        self._p, self._mu = 2.0 * u_1[1], 2.0 * u_1[0]  # 1111-1112: p = u_1.sub(1), mu = u_1.sub(0)
        if print_error:
            self.print_error()
        return self.last_ksp

    def incompressible_non_linear_solve(self, nullspace_p=None, *, space_p=None, P=None, solver_parameters=None,
                                        Multigrid=False, lambda_v_bounds=None, lambda_p_bounds=None,
                                        max_non_linear_iter=10, relative_non_linear_tol=10.0**-5,
                                        absolute_non_linear_tol=10.0**-8, print_error_linear=False,
                                        print_error_non_linear=True, create_output=False, plots=False, amg=None,
                                        amg_p=None):
        """control/control.py:1203-1486: Picard loop of stationary Navier-Stokes control."""
        if space_p is None:
            space_p = getattr(self, "_space_p", None)
            if space_p is None:
                raise ValueError("Undefined space_p")
        else:
            self.set_space_p(space_p)
        B = space_p["B"]
        n_p = space_p["M_p"].shape[0]
        v_old, zeta_old = self._v.copy(), self._zeta.copy()
        p_old = np.array(getattr(self, "_p", np.zeros(n_p)), dtype=float)
        mu_old = np.array(getattr(self, "_mu", np.zeros(n_p)), dtype=float)
        f = self._assembled_force()
        v_d = self._assembled_desired_state()

        r = None

        def residual():                                 # 1272-1319
            nonlocal r
            r00, r01 = self.non_linear_res_eval(v_d, f, v_old, zeta_old, self.construct_D_v(v_old))
            r00 = r00 - B.T @ mu_old
            r01 = r01 - B.T @ p_old
            self._bc(r00)
            self._bc(r01)
            r = r00, r01, -(B @ v_old), -(B @ zeta_old)
            return float(np.sqrt(sum(a @ a for a in r)))

        def step():
            nonlocal v_old, zeta_old, p_old, mu_old
            ksp = self.incompressible_linear_solve(nullspace_p, space_p=space_p, P=P, solver_parameters=solver_parameters,
                                                   Multigrid=Multigrid, lambda_v_bounds=lambda_v_bounds,
                                                   lambda_p_bounds=lambda_p_bounds, v_d=r[0], f=r[1], div_v=r[2],
                                                   div_zeta=r[3], print_error=print_error_linear, amg=amg, amg_p=amg_p)
            self.inner_iterations.append(ksp.its)
            v_old = v_old + self._v
            if self._bc_values is not None:
                v_old[self._bc_dofs] = self._bc_values
            zeta_old = zeta_old + self._zeta
            self._bc(zeta_old)
            p_old = p_old + self._p
            mu_old = mu_old + self._mu
            self._v, self._zeta, self._p, self._mu = v_old.copy(), zeta_old.copy(), p_old.copy(), mu_old.copy()
        self.non_linear_history, self.inner_iterations = [], []
        k = picard(residual, step, self.non_linear_history, max_iter=max_non_linear_iter,
                   rel_tol=relative_non_linear_tol, abs_tol=absolute_non_linear_tol, verbose=print_error_non_linear)
        if print_error_non_linear:
            self.print_error()
        return k

    # ------------------------------------------------------------------ non_linear_solve
    def non_linear_res_eval(self, v_d, f, v_old, zeta_old, D_v):
        """control/control.py:452-487."""
        M = self._M
        rhs_0 = v_d - M @ v_old - D_v.T @ zeta_old
        rhs_1 = f - D_v @ v_old + (1.0 / self._beta) * (M @ zeta_old)
        self._bc(rhs_0)
        self._bc(rhs_1)
        return rhs_0, rhs_1

    def non_linear_solve(self, *, P=None, solver_parameters=None, Multigrid=False, lambda_v_bounds=None,
                         max_non_linear_iter=10, relative_non_linear_tol=10.0**-5, absolute_non_linear_tol=10.0**-8,
                         print_error_linear=False, print_error_non_linear=True, create_output=False, plots=False, **amg):
        """control/control.py:630-800: Picard / Gauss-Newton loop; every outer iteration hands the new
        ``D_v`` values to the GPU and solves for the increment there."""
        v_old = self._v.copy()
        zeta_old = self._zeta.copy()
        f = self._assembled_force()
        v_d = self._assembled_desired_state()
        rhs_0 = rhs_1 = None

        def residual():
            nonlocal rhs_0, rhs_1
            rhs_0, rhs_1 = self.non_linear_res_eval(v_d, f, v_old, zeta_old, self.construct_D_v(v_old))
            return float(np.sqrt(rhs_0 @ rhs_0 + rhs_1 @ rhs_1))

        def step():
            nonlocal v_old, zeta_old
            self.linear_solve(P=P, solver_parameters=solver_parameters, Multigrid=Multigrid,
                              lambda_v_bounds=lambda_v_bounds, v_d=rhs_0, f=rhs_1, print_error=print_error_linear, **amg)
            v_old = v_old + self._v
            if self._bc_values is not None:             # 690-693
                v_old[self._bc_dofs] = self._bc_values
            zeta_old = zeta_old + self._zeta
            self._bc(zeta_old)
            self._v, self._zeta = v_old.copy(), zeta_old.copy()
        self.non_linear_history = []
        k = picard(residual, step, self.non_linear_history, max_iter=max_non_linear_iter,
                   rel_tol=relative_non_linear_tol, abs_tol=absolute_non_linear_tol, verbose=print_error_non_linear)
        if print_error_non_linear:
            self.print_error()
        return k
