"""Host-side mirror of ``Control.Instationary`` for the heat-control path (the caller of the
hot path: SURVEY.md section 8 rows a8, a11).

In the reference this layer is UFL/Firedrake: it builds the block dicts, assembles the
right-hand sides and drives ``MultiBlockSystem.solve`` (control/control.py:2820-3375) and the
Picard / Gauss-Newton loop (control/control.py:3377-3590, residual 2442-2818).  Here the same
driver works on ASSEMBLED objects -- the mass matrix, a callable returning the matrix of
``forward_form`` (or of its derivative) at a given state and time, nodal data tested against
the basis -- because only those ever reach the CUDA library.  Host work in this file is the
small vector algebra Firedrake does on the CPU in the reference (right-hand sides, residuals,
unpacking); every solve runs on the GPU through ``MultiBlockSystem``.

Keeps the reference's names, keyword arguments and defaults, including both spellings of the
force keyword (``force_function`` in the constructor, control/control.py:1490, ``force_f`` in
README.md:57 and every test).
"""
import numpy as np

from .system import MultiBlockSystem

__all__ = ["Control", "build_rhs"]


def _apply_T_1(x):      # control/control.py:26-41
    y = x.copy()
    y[:-1] += x[1:]
    return y


def _apply_T_2(x):      # control/control.py:44-59
    y = x.copy()
    y[1:] += x[:-1]
    return y


def build_rhs(M, K0, tau, n_t, CN, bc_dofs, v_d, f, v_0, check_v_d=True, check_f=True, bc_values=None,
              K_levels=None):
    """Right-hand sides of the heat-type rows (control/control.py:2990-3243; the Stokes driver
    builds its velocity rows the same way, 3961-4243).  ``v_d``, ``f``: (n_t, n) cofunction values
    (``M @ nodal``), or ready blocks (N, n) when the matching check_* is False; ``K0``: D_v at the
    initial condition.  ``bc_values`` (n_t, len(bc_dofs)): inhomogeneous, time-dependent Dirichlet
    data of the state, lifted into the right-hand sides as the reference does with ``v_inhom``
    (control/control.py:2993-3124 BE, 3137-3212 CN); ``K_levels``: D_v per time level for those terms
    (default: ``K0`` at every level).  Returns the final (T-transformed) ``b_0``, ``b_1`` of shape (N, n)."""
    n = M.shape[0]
    N = n_t - 1 if CN else n_t
    b_0 = np.zeros((N, n))
    b_1 = np.zeros((N, n))
    lift = None
    if bc_values is not None:
        lift = np.zeros((n_t, n))
        lift[:, bc_dofs] = np.asarray(bc_values, dtype=float)
    Kl = [K0] * n_t if K_levels is None else list(K_levels)

    def bc(b):
        b[..., bc_dofs] = 0.0
    if not CN:                                          # control.py:2990-3130
        if check_v_d:
            b_0[:n_t - 1] = tau * v_d[:n_t - 1]
            if lift is not None:
                b_0[:n_t - 1] -= tau * (M @ lift[:n_t - 1].T).T
            bc(b_0)
        else:
            b_0[:] = v_d
        if check_f:
            b_1[0] = tau * (K0 @ v_0) + M @ v_0
            b_1[1:] = tau * f[1:]
            if lift is not None:
                for i in range(n_t):
                    b_1[i] -= tau * (Kl[i] @ lift[i]) + M @ lift[i]
                    if i > 0:
                        b_1[i] += M @ lift[i - 1]
            bc(b_1)
        else:
            b_1[:] = f
    else:                                               # control.py:3131-3243
        if check_v_d:
            b_0[:] = 0.5 * tau * (v_d[:-1] + v_d[1:])
            if lift is not None:
                b_0[:] -= 0.5 * tau * (M @ lift[1:].T).T
                b_0[1:] -= 0.5 * tau * (M @ lift[1:-1].T).T
            bc(b_0)
            b_0[0] -= 0.5 * tau * (M @ v_0)
            bc(b_0[0])
        else:
            b_0[:] = v_d
        if check_f:
            b_1[:] = 0.5 * tau * (f[:-1] + f[1:])
            if lift is not None:
                for i in range(N):
                    b_1[i] -= 0.5 * tau * (Kl[i + 1] @ lift[i + 1]) + M @ lift[i + 1]
                    if i > 0:
                        b_1[i] -= 0.5 * tau * (Kl[i] @ lift[i]) - M @ lift[i]
            bc(b_1)
            b_1[0] -= 0.5 * tau * (K0 @ v_0) - M @ v_0
            bc(b_1[0])
        else:
            b_1[:] = f
        b_0 = _apply_T_1(b_0)
        b_1 = _apply_T_2(b_1)
    return b_0, b_1


class Control:
    class Instationary:
        def __init__(self, M, forward_matrix, *, desired_state=None, force_f=None, force_function=None,
                     beta=1.0e-3, Gauss_Newton=False, CN=True, n_t=20, initial_condition=None,
                     time_interval=(0.0, 1.0), bc_dofs=(), bc_values=None, device=None, rank=0, world=1,
                     block_size=1):
            """``M``: mass matrix (scipy CSR).  ``forward_matrix(v_i, t, gauss_newton)`` -> CSR
            on M's pattern: the matrix ``D_v`` of ``construct_D_v`` (control.py:1887-1896) at
            state ``v_i`` and time ``t``; a plain CSR matrix means a linear, time-independent
            operator.  ``desired_state(t)`` -> (M @ v_hat(t), v_hat(t)), the two returns of
            the reference's callable (control.py:1929-1931); ``force_f(t)`` -> M @ f(t).
            ``bc_values``: None (homogeneous Dirichlet data) or a callable ``t -> values at bc_dofs``
            (the reference's time-dependent ``bcs_v(space, t)``, control/control.py:1504-1530).
            ``block_size``: block size of the state space (``M.petscmat.getBlockSize()``; dofs interleaved as
            ``bs * node + comp``), passed to every device system this instance creates -- the heat-type system and
            the velocity system of the Stokes / Navier-Stokes solves -- whose preconditioners then run their time
            sweeps on the scalar block when the matrices are ``I_bs (x) S``.  One GPU only."""
            if force_f is not None and force_function is not None:
                raise TypeError("give either force_f or force_function")
            if int(block_size) not in (1, 2, 3):
                raise ValueError(f"block_size must be 1, 2 or 3, not {block_size}")
            if int(block_size) > 1 and world > 1:
                raise ValueError("block_size > 1 runs on one GPU: block-scalar sweeps are not available with world > 1")
            self._block_size = int(block_size)
            self._M = M.tocsr()
            self._forward_matrix = forward_matrix
            self._desired_state = desired_state
            self._force = force_f if force_f is not None else force_function
            self._beta = float(beta)
            self._Gauss_Newton = bool(Gauss_Newton)
            self._CN = bool(CN)
            self._n_t = int(n_t)
            self._time_interval = tuple(time_interval)
            self._bc_dofs = np.ascontiguousarray(bc_dofs, dtype=np.int32)
            self._bc_values = bc_values
            self._initial_condition = initial_condition
            self._n = self._M.shape[0]
            self._v = np.zeros((self._n_t, self._n))          # control.py:1569-1597
            self._zeta = np.zeros((self._n_t, self._n))
            self._system = None
            self._dev = dict(device=device, rank=rank, world=world)
            self.last_ksp = None
            self.non_linear_history = []

        # ------------------------------------------------------------------ helpers
        @property
        def tau(self):
            t_0, T_f = self._time_interval
            return (T_f - t_0) / (self._n_t - 1.0)

        def _times(self):
            return self._time_interval[0] + self.tau * np.arange(self._n_t)

        def _is_linear(self):
            return not callable(self._forward_matrix)

        def construct_D_v(self, v_i, t):
            if self._is_linear():
                return self._forward_matrix
            return self._forward_matrix(v_i, t, self._Gauss_Newton)

        def _K_levels(self, v):
            if self._is_linear():
                return self._forward_matrix
            return [self.construct_D_v(v[i], t) for i, t in enumerate(self._times())]

        def construct_f(self):          # control.py:1898-1916
            if self._force is None:
                return np.zeros((self._n_t, self._n))
            return np.stack([self._force(t) for t in self._times()])

        def construct_v_d(self):        # control.py:1918-1941
            if self._desired_state is None:
                self._true_v = np.zeros((self._n_t, self._n))
                return np.zeros((self._n_t, self._n))
            pairs = [self._desired_state(t) for t in self._times()]
            self._true_v = np.stack([p[1] for p in pairs])
            return np.stack([p[0] for p in pairs])

        def _bc(self, b):
            b[..., self._bc_dofs] = 0.0

        def _ensure_system(self, K):
            if self._system is None:
                self._system = MultiBlockSystem(self._M, K, n_t=self._n_t, beta=self._beta, CN=self._CN,
                                                time_interval=self._time_interval, bc_dofs=self._bc_dofs,
                                                **self._block_kw("block_size"), **self._dev)
                if self._dev["world"] > 1:
                    self._system.init_comm()
            else:
                self._system.set_K(K)
            return self._system

        def _block_kw(self, name):
            # the block size only travels when it is not the default, so stand-in systems need not know it
            return {name: self._block_size} if self._block_size != 1 else {}

        def close(self):
            if self._system is not None:
                self._system.close()
                self._system = None
            if getattr(self, "_stokes", None) is not None:
                self._stokes.close()
                self._stokes = None

        def _dirichlet_data(self):
            """(n_t, len(bc_dofs)) boundary values of the state per time level, or None."""
            if self._bc_values is None:
                return None
            return np.stack([np.asarray(self._bc_values(t), dtype=float) for t in self._times()])

        def _build_rhs(self, v_0, v_d, f, K0, check_v_d, check_f, K_levels=None):
            return build_rhs(self._M, K0, self.tau, self._n_t, self._CN, self._bc_dofs, v_d, f, v_0,
                             check_v_d=check_v_d, check_f=check_f, bc_values=self._dirichlet_data(),
                             K_levels=K_levels)

        # ------------------------------------------------------------------ linear_solve
        def linear_solve(self, *, P=None, solver_parameters=None, Multigrid=False, lambda_v_bounds=None,
                         v_d=None, f=None, print_error=True, create_output=False, plots=False,
                         pc_mode="triangular", **amg):
            """control/control.py:2820-3375 (homogeneous Dirichlet data)."""
            n_t, n, tau, CN = self._n_t, self._n, self.tau, self._CN
            M = self._M
            N = n_t - 1 if CN else n_t
            v_0 = np.zeros(n) if self._initial_condition is None else np.asarray(self._initial_condition, float)
            check_f, check_v_d = f is None, v_d is None
            if check_f:
                f = self.construct_f()
            if check_v_d:
                v_d = self.construct_v_d()
            K = self._K_levels(self._v)                         # D_v at self._v, control.py:2884-2904
            K0 = K if self._is_linear() else self.construct_D_v(v_0, self._time_interval[0])
            b_0, b_1 = self._build_rhs(v_0, v_d, f, K0, check_v_d, check_f,
                                       K_levels=None if self._is_linear() else K)
            if solver_parameters is None:                       # control.py:3260-3266
                solver_parameters = {"linear_solver": "gmres", "gmres_restart": 10, "maximum_iterations": 50,
                                     "relative_tolerance": 1.0e-6, "absolute_tolerance": 0.0,
                                     "monitor_convergence": print_error}
            system = self._ensure_system(K)
            if P is None:                                       # control.py:3245-3258
                system.setup_preconditioner(lambda_v_bounds=lambda_v_bounds, Multigrid=Multigrid,
                                            mode=pc_mode, **amg)
                pc_fn = "builtin"
            else:
                pc_fn = P
            rows = slice(system.row_begin, system.row_begin + system.n_local)
            v = np.zeros((N, system.n_local))
            zeta = np.zeros((N, system.n_local))
            self.last_ksp = system.solve(v, zeta, np.ascontiguousarray(b_0[:, rows]),
                                         np.ascontiguousarray(b_1[:, rows]),
                                         solver_parameters=solver_parameters, pc_fn=pc_fn)
            if system.world > 1:
                v, zeta = system.allgather_blocks(v), system.allgather_blocks(zeta)
            if CN:                                              # control.py:3299-3312
                v_new = np.zeros((n_t, n))
                zeta_new = np.zeros((n_t, n))
                if check_f and check_v_d:
                    v_new[0] = v_0
                v_new[1:] = v
                zeta_new[:-1] = zeta
                self._v, self._zeta = v_new, zeta_new
            else:
                self._v, self._zeta = v, zeta
            self._bc(self._zeta)                                # set_zeta re-applies bcs, control.py:1847-1856
            g = self._dirichlet_data()
            if g is not None:                                   # set_v re-applies the (inhomogeneous) bcs, 1836-1845
                self._v[:, self._bc_dofs] = g
            return self.last_ksp

        # ------------------------------------------------------------------ Stokes control
        def set_space_p(self, space_p):
            """``space_p``: the assembled objects of the pressure space, a dict with the divergence
            matrix ``B`` (n_p x n_v, ``-inner(div(v_trial), p_test) * dx``), the pressure mass
            matrix ``M_p`` and the pressure Laplacian ``K_p`` (control/control.py:3709, 3746-3747).
            Optional ``forward_matrix_p(v_i, t, gauss_newton)`` -> CSR on M_p's pattern: the forward form
            on the pressure space at the velocity state ``v_i`` (``D_p_i``, control/control.py:3787-3789);
            needed when the forward operator is not the Stokes one (Navier-Stokes Picard iterations)."""
            self._space_p = space_p

        def incompressible_linear_solve(self, nullspace_p=None, *, space_p=None, P=None, solver_parameters=None,
                                        Multigrid=False, lambda_v_bounds=None, lambda_p_bounds=None, v_d=None,
                                        f=None, div_v=None, div_zeta=None, print_error=True, create_output=False,
                                        plots=False, amg=None, amg_p=None):
            """control/control.py:3592-4725 (Dirichlet velocity data homogeneous or, through ``bc_values``
            of the constructor, inhomogeneous and time dependent; a callable forward matrix is evaluated
            at the current ``_v`` per time level, with ``space_p["forward_matrix_p"]`` on the pressure space).  ``nullspace_p``: None or "constant" -- the pressure blocks
            carry ConstantNullspace as in every caller of the reference (test/test_control.py,
            README.md).  Sets ``_v``, ``_zeta``, ``_p``, ``_mu`` and returns the KSP information."""
            from .stokes import StokesSystem
            if space_p is None:
                space_p = getattr(self, "_space_p", None)
                if space_p is None:
                    raise ValueError("Undefined space_p")               # control.py:3604-3609
            else:
                self.set_space_p(space_p)
            if nullspace_p not in (None, "constant"):
                raise ValueError("only the constant pressure nullspace is supported")
            n_t, n, tau, CN = self._n_t, self._n, self.tau, self._CN
            N = n_t - 1 if CN else n_t
            n_p = space_p["M_p"].shape[0]
            v_0 = np.zeros(n) if self._initial_condition is None else np.asarray(self._initial_condition, float)
            check_f, check_v_d = f is None, v_d is None
            if check_f:
                f = self.construct_f()
            if check_v_d:
                v_d = self.construct_v_d()
            K = self._K_levels(self._v)                             # D_v_i at the current state, 3780-3785
            D_p = None
            if self._is_linear():
                K0 = K
            else:
                K0 = self.construct_D_v(v_0, self._time_interval[0])
                fp = space_p.get("forward_matrix_p")
                if fp is None:
                    raise ValueError("a non-linear forward operator needs space_p['forward_matrix_p']")
                D_p = [fp(self._v[i], t, self._Gauss_Newton) for i, t in enumerate(self._times())]      # 3787-3789
            b_0_0, b_0_1 = self._build_rhs(v_0, v_d, f, K0, check_v_d, check_f,
                                           K_levels=None if self._is_linear() else K)  # 3961-4243
            b_1_0 = np.zeros((N, n_p)) if div_v is None else np.array(div_v, dtype=float)      # 4107-4128, 4207-4228
            g = self._dirichlet_data()
            if div_v is None and g is not None:                 # b_1_0[i] -= tau B v_inhom (4107-4119, 4207-4219)
                lift = np.zeros((n_t, n))
                lift[:, self._bc_dofs] = g
                b_1_0 -= tau * (space_p["B"] @ (lift[1:] if CN else lift).T).T
            b_1_1 = np.zeros((N, n_p)) if div_zeta is None else np.array(div_zeta, dtype=float)
            if CN:                                                                        # 4233-4234
                b_1_0 = _apply_T_2(b_1_0)
                b_1_1 = _apply_T_1(b_1_1)
            b_0 = np.concatenate([b_0_0, b_0_1])
            b_1 = np.concatenate([b_1_0, b_1_1])
            if solver_parameters is None:                                                 # 4291-4297
                solver_parameters = {"linear_solver": "fgmres", "fgmres_restart": 10, "maximum_iterations": 100,
                                     "relative_tolerance": 1.0e-6, "absolute_tolerance": 0.0,
                                     "monitor_convergence": print_error}
            if getattr(self, "_stokes", None) is None:
                self._stokes = StokesSystem(self._M, K, space_p["B"], space_p["M_p"], space_p["K_p"], n_t=n_t,
                                            beta=self._beta, CN=CN, time_interval=self._time_interval,
                                            bc_dofs_v=self._bc_dofs, device=self._dev["device"], D_p=D_p,
                                            **self._block_kw("velocity_block_size"))
            elif not self._is_linear():
                self._stokes.set_forward(K, D_p)
            system = self._stokes
            if P is None:                                           # control.py:4686-4689: pc_fn = P or the in-built one
                system.setup_preconditioner(lambda_v_bounds=lambda_v_bounds, lambda_p_bounds=lambda_p_bounds, amg=amg,
                                            amg_p=amg_p, Multigrid=Multigrid)
            u_0 = np.zeros((2 * N, n))
            u_1 = np.zeros((2 * N, n_p))
            self.last_ksp = system.solve(u_0, u_1, b_0, b_1, solver_parameters=solver_parameters,
                                         pc_fn="builtin" if P is None else P)
            if solver_parameters.get("monitor_convergence", True):
                for it, r_norm in enumerate(self.last_ksp.history):
                    print(f"KSP: iteration {it:d}, residual norm {r_norm:.16e}")
            if CN:                                                                        # 4705-4716
                v_new = np.zeros((n_t, n))
                zeta_new = np.zeros((n_t, n))
                if check_f and check_v_d:
                    v_new[0] = v_0
                v_new[1:] = u_0[:N]
                zeta_new[:-1] = u_0[N:]
                self._v, self._zeta = v_new, zeta_new
            else:                                                                         # 4717-4725
                self._v, self._zeta = u_0[:N].copy(), u_0[N:].copy()
            self._p, self._mu = u_1[N:].copy(), u_1[:N].copy()
            self._bc(self._zeta)
            if g is not None:                                   # set_v re-applies the (inhomogeneous) bcs
                self._v[:, self._bc_dofs] = g
            return self.last_ksp

        def incompressible_non_linear_solve(self, nullspace_p=None, *, space_p=None, P=None, solver_parameters=None,
                                            Multigrid=False, lambda_v_bounds=None, lambda_p_bounds=None,
                                            max_non_linear_iter=10, relative_non_linear_tol=10.0**-5,
                                            absolute_non_linear_tol=10.0**-8, print_error_linear=False,
                                            print_error_non_linear=True, create_output=False, plots=False,
                                            amg=None, amg_p=None, device_loop=None):
            """control/control.py:4886-5219: Picard loop of Navier-Stokes control.  Every outer iteration
            re-linearises the forward operator around the new velocity on both spaces, hands the values to
            the GPU and solves the outer Stokes-type system for the increment there.

            ``device_loop``: True keeps the iterate, the residual and the increments in HBM
            (``_incompressible_non_linear_solve_device``; in-built preconditioner only, so ``P=`` raises
            ``ValueError``); False or None runs the host loop, which evaluates the residual on the host and moves the
            whole outer vector both ways every iteration.  None stays the host loop for now because the stand-in
            systems that exercise both loops on inhomogeneous data have no device methods."""
            if device_loop and P is not None:
                raise ValueError("device_loop=True runs the in-built preconditioner; it does not take P=")
            if space_p is None:
                space_p = getattr(self, "_space_p", None)
                if space_p is None:
                    raise ValueError("Undefined space_p")               # 4904-4910
            else:
                self.set_space_p(space_p)
            n_t, n, tau, CN = self._n_t, self._n, self.tau, self._CN
            N = n_t - 1 if CN else n_t
            B = space_p["B"]
            n_p = space_p["M_p"].shape[0]
            v_old = self._v.copy()
            zeta_old = self._zeta.copy()
            p_old = np.array(getattr(self, "_p", np.zeros((N, n_p))), dtype=float)
            mu_old = np.array(getattr(self, "_mu", np.zeros((N, n_p))), dtype=float)
            v_0 = np.zeros(n) if self._initial_condition is None else np.asarray(self._initial_condition, float)
            if CN:
                v_old[0] = v_0                                          # 4968-4969
            zeta_old[n_t - 1] = 0.0
            f = self.construct_f()
            v_d = self.construct_v_d()
            g = self._dirichlet_data()
            self._v, self._zeta = v_old.copy(), zeta_old.copy()
            if device_loop:
                if nullspace_p not in (None, "constant"):
                    raise ValueError("only the constant pressure nullspace is supported")
                return self._incompressible_non_linear_solve_device(
                    space_p, v_old, zeta_old, p_old, mu_old, v_0, v_d, f, g, solver_parameters, Multigrid,
                    lambda_v_bounds, lambda_p_bounds, max_non_linear_iter, relative_non_linear_tol,
                    absolute_non_linear_tol, print_error_linear, print_error_non_linear, amg, amg_p)

            def res_eval():                                             # 4979-5072
                r00, r01 = self.non_linear_res_eval(v_old, zeta_old, v_0, v_d, f)
                r00 -= tau * (B.T @ mu_old.T).T
                r01 -= tau * (B.T @ p_old.T).T
                self._bc(r00)
                self._bc(r01)
                r10 = -(B @ (v_old[1:] if CN else v_old).T).T
                r11 = -(B @ (zeta_old[:-1] if CN else zeta_old).T).T
                return r00, r01, r10, r11

            def norm(parts):
                return float(np.sqrt(sum((a ** 2).sum() for a in parts)))

            r = res_eval()
            norm_0 = norm(r)
            norm_k, k = norm_0, 0
            self.non_linear_history = [norm_0]
            self.inner_iterations = []
            if print_error_non_linear:
                print(f"Initial non-linear residual: {norm_0:.16e}")
            while norm_k > relative_non_linear_tol * norm_0 and norm_k > absolute_non_linear_tol:
                ksp = self.incompressible_linear_solve(nullspace_p, space_p=space_p, P=P,
                                                       solver_parameters=solver_parameters, Multigrid=Multigrid,
                                                       lambda_v_bounds=lambda_v_bounds, lambda_p_bounds=lambda_p_bounds,
                                                       v_d=r[0], f=r[1], div_v=tau * r[2], div_zeta=tau * r[3],
                                                       print_error=print_error_linear, amg=amg, amg_p=amg_p)
                self.inner_iterations.append(ksp.its)
                v_old = v_old + self._v                                 # 5127-5160
                if g is not None:
                    v_old[:, self._bc_dofs] = g
                p_old = p_old + self._p
                zeta_old = zeta_old + self._zeta
                self._bc(zeta_old)
                mu_old = mu_old + self._mu
                self._v, self._zeta = v_old.copy(), zeta_old.copy()
                self._p, self._mu = p_old.copy(), mu_old.copy()
                r = res_eval()
                norm_k = norm(r)
                k += 1
                self.non_linear_history.append(norm_k)
                if print_error_non_linear:
                    print(f"Non-linear solver: iteration {k:d}, non-linear residual norm {norm_k:.16e}")
                if k + 1 > max_non_linear_iter:
                    break
            return k

        def _incompressible_non_linear_solve_device(self, space_p, v_old, zeta_old, p_old, mu_old, v_0, v_d, f, g,
                                                    solver_parameters, Multigrid, lambda_v_bounds, lambda_p_bounds,
                                                    max_non_linear_iter, rel_tol, abs_tol, print_error_linear,
                                                    print_error_non_linear, amg, amg_p):
            """The loop of control/control.py:4886-5219 with device-resident iterates.  The right-hand side of the
            data is built once (velocity rows as ``incompressible_linear_solve`` builds them, pressure rows zero).
            Per outer iteration: the increment solve reads the residual where it lies, the velocity state goes to the
            host (N n_v doubles) for the assembly of ``D_v_i`` / ``D_p_i``, their values come back
            (``set_forward``), a copy of b is lifted with g (``lift_bc_device``), and the residual is
            ``ctl_stokes_nonlinear_residual``: b - A_raw x with the RAW coupling products, as ``res_eval`` has them
            (no ConstantNullspace corrections), and the norm of its untransformed parts."""
            from .stokes import StokesSystem
            n_t, tau, CN = self._n_t, self.tau, self._CN
            N = n_t - 1 if CN else n_t
            n_p = space_p["M_p"].shape[0]
            times = self._times()
            bd = self._bc_dofs
            linear = self._is_linear()
            fp = space_p.get("forward_matrix_p")
            if not linear and fp is None:
                raise ValueError("a non-linear forward operator needs space_p['forward_matrix_p']")

            def forward(v):                                             # D_v_i, D_p_i at the state, 3780-3789
                if linear:
                    return self._forward_matrix, None
                return ([self.construct_D_v(v[i], t) for i, t in enumerate(times)],
                        [fp(v[i], t, self._Gauss_Newton) for i, t in enumerate(times)])

            def rhs(v_init):                                            # 3961-4243, homogeneous data
                K0 = self._forward_matrix if linear else self.construct_D_v(v_init, self._time_interval[0])
                b_0_0, b_0_1 = build_rhs(self._M, K0, tau, n_t, CN, bd, v_d, f, v_init)
                return system.to_device(np.concatenate([b_0_0, b_0_1]), np.zeros((2 * N, n_p)))
            if solver_parameters is None:                               # 4291-4297
                solver_parameters = {"linear_solver": "fgmres", "fgmres_restart": 10, "maximum_iterations": 100,
                                     "relative_tolerance": 1.0e-6, "absolute_tolerance": 0.0,
                                     "monitor_convergence": print_error_linear}
            K, D_p = forward(v_old)
            if getattr(self, "_stokes", None) is None:
                self._stokes = StokesSystem(self._M, K, space_p["B"], space_p["M_p"], space_p["K_p"], n_t=n_t,
                                            beta=self._beta, CN=CN, time_interval=self._time_interval,
                                            bc_dofs_v=bd, device=self._dev["device"], D_p=D_p,
                                            **self._block_kw("velocity_block_size"))
            elif not linear:
                self._stokes.set_forward(K, D_p)
            system = self._stokes
            if g is None:
                b_dev = b_hom = rhs(v_0)
            else:
                b_hom, b_dev = self._lifted_rhs_pair(system, rhs, v_old, v_0, g)
            x_dev = system.to_device(np.concatenate([v_old[1:], zeta_old[:-1]] if CN else [v_old, zeta_old]),
                                     np.concatenate([mu_old, p_old]))
            r_dev = system.new_vector()
            norm_0 = system.nonlinear_residual(b_dev, x_dev, r_dev)
            norm_k, k = norm_0, 0
            self.non_linear_history = [norm_0]
            self.inner_iterations = []
            if print_error_non_linear:
                print(f"Initial non-linear residual: {norm_0:.16e}")
            while norm_k > rel_tol * norm_0 and norm_k > abs_tol:
                system.setup_preconditioner(lambda_v_bounds=lambda_v_bounds, lambda_p_bounds=lambda_p_bounds, amg=amg,
                                            amg_p=amg_p, Multigrid=Multigrid)
                d_dev = system.new_vector()
                self.last_ksp = system.solve_device(r_dev, d_dev, solver_parameters=solver_parameters)
                if not solver_parameters.get("preconditioner", False) and self.last_ksp.reason <= 0:
                    raise RuntimeError("Solver failed to converge")
                if solver_parameters.get("monitor_convergence", True):
                    for it, r_norm in enumerate(self.last_ksp.history):
                        print(f"KSP: iteration {it:d}, residual norm {r_norm:.16e}")
                self.inner_iterations.append(self.last_ksp.its)
                x_dev += d_dev
                v_blocks = system.velocity_state_to_host(x_dev)
                if CN:
                    v_old[1:] = v_blocks
                else:
                    v_old = v_blocks
                if g is not None:                                       # 5127-5160
                    v_old[:, bd] = g
                if not linear:
                    system.set_forward(*forward(v_old))
                if g is not None:
                    b_dev = system.lift_bc_device(g, b_hom.clone())
                norm_k = system.nonlinear_residual(b_dev, x_dev, r_dev)
                k += 1
                self.non_linear_history.append(norm_k)
                if print_error_non_linear:
                    print(f"Non-linear solver: iteration {k:d}, non-linear residual norm {norm_k:.16e}")
                if k + 1 > max_non_linear_iter:
                    break
            x_0, x_1 = system.to_host_blocks(x_dev)
            if CN:
                v_old[1:], zeta_old[:-1] = x_0[:N], x_0[N:]
            else:
                v_old, zeta_old = x_0[:N].copy(), x_0[N:].copy()
            if k > 0:
                if g is not None:
                    v_old[:, bd] = g
                self._bc(zeta_old)
            self._v, self._zeta = v_old.copy(), zeta_old.copy()
            self._p, self._mu = x_1[N:].copy(), x_1[:N].copy()
            return k

        # ------------------------------------------------------------------ non_linear_solve
        def non_linear_res_eval(self, v_old, zeta_old, v_0, v_d, f):
            """control/control.py:2442-2818: right-hand side minus the KKT operator applied to
            the current iterate, row by row, with D_v evaluated at the iterate."""
            n_t, n, tau, beta, CN, M = self._n_t, self._n, self.tau, self._beta, self._CN, self._M
            times = self._times()
            D = [self.construct_D_v(v_old[i], times[i]) for i in range(n_t)]
            if CN:
                h = 0.5 * tau
                rhs_0 = np.zeros((n_t - 1, n))
                rhs_1 = np.zeros((n_t - 1, n))
                for i in range(n_t - 1):                        # control.py:2621-2814
                    rhs_0[i] = h * (v_d[i] + v_d[i + 1]) - h * (M @ v_old[i]) - h * (M @ v_old[i + 1]) \
                        - (h * (D[i].T @ zeta_old[i]) + M @ zeta_old[i]) \
                        - (h * (D[i + 1].T @ zeta_old[i + 1]) - M @ zeta_old[i + 1])
                    rhs_1[i] = h * (f[i] + f[i + 1]) - (h * (D[i] @ v_old[i]) - M @ v_old[i]) \
                        - (h * (D[i + 1] @ v_old[i + 1]) + M @ v_old[i + 1]) \
                        + (h / beta) * (M @ zeta_old[i]) + (h / beta) * (M @ zeta_old[i + 1])
            else:
                rhs_0 = np.zeros((n_t, n))
                rhs_1 = np.zeros((n_t, n))
                D_v_0 = self.construct_D_v(v_0, times[0])
                for i in range(n_t):                            # control.py:2457-2620
                    if i < n_t - 1:
                        rhs_0[i] = tau * v_d[i] - tau * (M @ v_old[i]) \
                            - (tau * (D[i].T @ zeta_old[i]) + M @ zeta_old[i]) + M @ zeta_old[i + 1]
                    else:
                        rhs_0[i] = -(tau * (D[i].T @ zeta_old[i]) + M @ zeta_old[i])
                    if i == 0:
                        rhs_1[0] = (tau * (D_v_0 @ v_0) + M @ v_0) - (tau * (D[0] @ v_old[0]) + M @ v_old[0])
                    else:
                        rhs_1[i] = tau * f[i] - (tau * (D[i] @ v_old[i]) + M @ v_old[i]) + M @ v_old[i - 1] \
                            + (tau / beta) * (M @ zeta_old[i])
            self._bc(rhs_0)
            self._bc(rhs_1)
            return rhs_0, rhs_1

        def non_linear_solve(self, *, P=None, solver_parameters=None, Multigrid=False, lambda_v_bounds=None,
                             max_non_linear_iter=10, relative_non_linear_tol=10.0**-5,
                             absolute_non_linear_tol=10.0**-8, print_error_linear=False,
                             print_error_non_linear=True, create_output=False, plots=False, device_loop=None, **amg):
            """control/control.py:3377-3590: Picard / Gauss-Newton loop.  Every outer iteration
            hands new ``K_i`` values to the GPU (``MultiBlockSystem.set_K``) and solves for
            the increment.

            ``device_loop``: True keeps the iterate, the residual and the increments in HBM
            (``_non_linear_solve_device``), with homogeneous or inhomogeneous Dirichlet data; it needs the in-built
            preconditioner and one rank, so ``P=`` or ``world > 1`` raise ``ValueError``.  False runs the host loop.
            None keeps the device loop for homogeneous data, the in-built preconditioner, one rank and a non-linear
            forward operator, and the host loop otherwise: the stand-in systems that exercise both loops on
            inhomogeneous data have no device methods."""
            if device_loop and P is not None:
                raise ValueError("device_loop=True runs the in-built preconditioner; it does not take P=")
            if device_loop and self._dev["world"] > 1:
                raise ValueError("device_loop=True runs on one rank")
            n_t, n = self._n_t, self._n
            g = self._dirichlet_data()
            v_old = self._v.copy()
            zeta_old = self._zeta.copy()
            v_0 = np.zeros(n) if self._initial_condition is None else np.asarray(self._initial_condition, float)
            if self._CN:
                v_old[0] = v_0
            zeta_old[n_t - 1] = 0.0
            f = self.construct_f()
            v_d = self.construct_v_d()
            self._v, self._zeta = v_old.copy(), zeta_old.copy()
            if device_loop is None:
                device_loop = P is None and g is None and self._dev["world"] == 1 and not self._is_linear()
            if device_loop:
                # the iterate, the residual and the increments stay in HBM; only the state crosses the boundary,
                # because the forward form D_v(v_i) is assembled on the caller's side (Firedrake's) of it
                return self._non_linear_solve_device(v_old, zeta_old, v_0, v_d, f, solver_parameters, Multigrid,
                                                     lambda_v_bounds, max_non_linear_iter, relative_non_linear_tol,
                                                     absolute_non_linear_tol, print_error_linear,
                                                     print_error_non_linear, amg)
            rhs_0, rhs_1 = self.non_linear_res_eval(v_old, zeta_old, v_0, v_d, f)
            norm_0 = float(np.sqrt((rhs_0 ** 2).sum() + (rhs_1 ** 2).sum()))
            norm_k = norm_0
            k = 0
            self.non_linear_history = [norm_0]
            if print_error_non_linear:
                print(f"Initial non-linear residual: {norm_0:.16e}")
            while norm_k > relative_non_linear_tol * norm_0 and norm_k > absolute_non_linear_tol:
                self.linear_solve(P=P, solver_parameters=solver_parameters, Multigrid=Multigrid,
                                  lambda_v_bounds=lambda_v_bounds, v_d=rhs_0, f=rhs_1,
                                  print_error=print_error_linear, **amg)
                v_old = v_old + self._v
                if g is not None:                               # control.py:3480-3483
                    v_old[:, self._bc_dofs] = g
                zeta_old = zeta_old + self._zeta
                self._bc(zeta_old)
                self._v, self._zeta = v_old.copy(), zeta_old.copy()
                rhs_0, rhs_1 = self.non_linear_res_eval(v_old, zeta_old, v_0, v_d, f)
                norm_k = float(np.sqrt((rhs_0 ** 2).sum() + (rhs_1 ** 2).sum()))
                k += 1
                self.non_linear_history.append(norm_k)
                if print_error_non_linear:
                    print(f"Non-linear solver: iteration {k:d}, non-linear residual norm {norm_k:.16e}")
                if k + 1 > max_non_linear_iter:
                    break
            return k


        def _non_linear_solve_device(self, v_old, zeta_old, v_0, v_d, f, solver_parameters, Multigrid, lambda_v_bounds,
                                     max_non_linear_iter, rel_tol, abs_tol, print_error_linear, print_error_non_linear,
                                     amg):
            """The loop of control/control.py:3377-3525 with device-resident iterates.  Per outer iteration: the
            state goes to the host (D2H of one half vector) for the assembly of the ``D_v_i``, their values come
            back (``set_K``), the residual is ``ctl_nonlinear_residual`` (right-hand side of ``linear_solve`` for
            the data, built ONCE, minus the fused operator at the iterate: the identity of
            tests/test_oracle.py::test_non_linear_residual_is_rhs_minus_operator), and the increment solve reads
            it where it lies.  Inhomogeneous Dirichlet data g (INTEGRATION.md section 6): the residual takes a copy
            of b lifted with the K_i of the iterate (``lift_bc_device``), and g is written into the iterate."""
            n_t, n, CN = self._n_t, self._n, self._CN
            times = self._times()
            g = self._dirichlet_data()
            bd = self._bc_dofs

            def rhs(v_init):
                K0 = self.construct_D_v(v_init, self._time_interval[0])
                return system.to_device(*build_rhs(self._M, K0, self.tau, n_t, CN, bd, v_d, f, v_init))
            if solver_parameters is None:                       # control.py:3260-3266
                solver_parameters = {"linear_solver": "gmres", "gmres_restart": 10, "maximum_iterations": 50,
                                     "relative_tolerance": 1.0e-6, "absolute_tolerance": 0.0,
                                     "monitor_convergence": print_error_linear}
            system = self._ensure_system([self.construct_D_v(v_old[i], times[i]) for i in range(n_t)])
            if g is None:
                b_dev = rhs(v_0)
            else:
                b_hom, b_dev = self._lifted_rhs_pair(system, rhs, v_old, v_0, g)
            x_dev = system.to_device(*((v_old[1:], zeta_old[:-1]) if CN else (v_old, zeta_old)))
            r_dev = system.new_vector()
            norm_0 = system.nonlinear_residual(b_dev, x_dev, r_dev)
            norm_k, k = norm_0, 0
            self.non_linear_history = [norm_0]
            if print_error_non_linear:
                print(f"Initial non-linear residual: {norm_0:.16e}")
            while norm_k > rel_tol * norm_0 and norm_k > abs_tol:
                system.setup_preconditioner(lambda_v_bounds=lambda_v_bounds, Multigrid=Multigrid, **amg)
                d_dev = system.new_vector()
                self.last_ksp = system.solve_device(r_dev, d_dev, solver_parameters=solver_parameters, pc="builtin")
                if solver_parameters.get("monitor_convergence", True):
                    for it, r_norm in enumerate(self.last_ksp.history):
                        print(f"KSP: iteration {it:d}, residual norm {r_norm:.16e}")
                if not solver_parameters.get("preconditioner", False) and self.last_ksp.reason <= 0:
                    raise RuntimeError("Solver failed to converge")
                x_dev += d_dev
                v_blocks = system.to_host_blocks(x_dev)[0]
                if CN:
                    v_old[1:] = v_blocks
                else:
                    v_old = v_blocks.copy()
                if g is not None:                               # control.py:3480-3483
                    v_old[:, bd] = g
                system.set_K([self.construct_D_v(v_old[i], times[i]) for i in range(n_t)])
                if g is not None:
                    b_dev = system.lift_bc_device(g, b_hom.clone())
                norm_k = system.nonlinear_residual(b_dev, x_dev, r_dev)
                k += 1
                self.non_linear_history.append(norm_k)
                if print_error_non_linear:
                    print(f"Non-linear solver: iteration {k:d}, non-linear residual norm {norm_k:.16e}")
                if k + 1 > max_non_linear_iter:
                    break
            x_0, x_1 = system.to_host_blocks(x_dev)
            if CN:
                v_old[1:], zeta_old[:-1] = x_0, x_1
            else:
                v_old, zeta_old = x_0.copy(), x_1.copy()
            if g is not None and k > 0:
                v_old[:, bd] = g
            self._bc(zeta_old)
            self._v, self._zeta = v_old.copy(), zeta_old.copy()
            return k

        def _lifted_rhs_pair(self, system, rhs, v_old, v_0, g):
            """Device right-hand sides of a non-linear loop with inhomogeneous Dirichlet data g: the homogeneous b that
            every residual after the first lifts a copy of (for CN its initial condition is v_0 with g_0 on the
            boundary, because the loop writes g into every level of the iterate, level 0 included), and the b of the
            first residual, lifted with the boundary values the starting iterate carries.  ``rhs(v_init)`` builds a
            homogeneous device right-hand side."""
            b_first = rhs(v_0)
            b_hom = b_first
            if self._CN:
                v_0g = v_0.copy()
                v_0g[self._bc_dofs] = g[0]
                b_hom = rhs(v_0g)
            g_it = np.ascontiguousarray(v_old[:, self._bc_dofs])
            if np.any(g_it):
                b_first = system.lift_bc_device(g_it, b_first.clone())
            return b_hom, b_first


from .stationary import Stationary as _Stationary  # noqa: E402

Control.Stationary = _Stationary            # control/control.py:100 (heat-type drivers; N = 1 case of the same handle)
