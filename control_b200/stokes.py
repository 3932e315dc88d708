"""Host-side mirror of the outer block system of instationary Stokes control.

``StokesSystem`` plays the role of the ``MultiBlockSystem`` the reference builds in
``Control.Instationary.incompressible_linear_solve`` (control/control.py:3592-4725, system
construction at 4273-4289): block_00 = the heat-type KKT system on the velocity space,
block_01 / block_10 = diag(tau B^T) / diag(tau B), block_11 = None, with sub-block T
transforms (preconditioner/preconditioner.py:471-525), DirichletBCNullspace on the velocity
blocks and ConstantNullspace on the pressure blocks.  It is constructed from the five
spatial matrices the blocks are made of; every numeric operation runs in libctl_b200.so.

Vectors at this boundary are block-major: ``x_0`` of shape (2N, n_v) = [v | zeta] and ``x_1``
of shape (2N, n_p) = [mu | p], or one flat device vector [x_0 | x_1].
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L
from .system import KSPInfo, MultiBlockSystem, _as_host_f64, csr_arrays

__all__ = ["StokesSystem"]


class StokesSystem:
    def __init__(self, M_v, K_v, B, M_p, K_p, *, n_t, beta, CN, time_interval=(0.0, 1.0), bc_dofs_v=(),
                 epsilon=1e-3, device=None, D_p=None, velocity_block_size=1):
        """``K_v``: the forward matrix on the velocity space (one matrix or n_t matrices ``D_v_i``).  ``K_p``: the
        pressure Laplacian ``solver_K_p`` inverts (control/control.py:3746, 4300-4309).  ``D_p``: the forward
        form on the PRESSURE space (``D_p_i``, control/control.py:3787-3789; one matrix or n_t matrices) of the
        pressure-space KKT multiply; default ``K_p`` (the Stokes forward operator).  ``velocity_block_size``: block
        size of the velocity space (2 for a 2-D ``VectorFunctionSpace``): the velocity sweeps then run on the scalar
        block of ``I_2 (x) S`` (``MultiBlockSystem(block_size=)``)."""
        self.velocity = MultiBlockSystem(M_v, K_v, n_t=n_t, beta=beta, CN=CN, time_interval=time_interval,
                                         bc_dofs=bc_dofs_v, epsilon=epsilon, device=device,
                                         block_size=velocity_block_size)
        self.pressure = MultiBlockSystem(M_p, K_p if D_p is None else D_p, n_t=n_t, beta=beta, CN=CN,
                                         time_interval=time_interval, bc_dofs=(), epsilon=epsilon,
                                         device=self.velocity.device.index, stream=self.velocity.stream)
        self._K_p_solver = None if D_p is None else np.ascontiguousarray(self.pressure._same_pattern(K_p))
        self._lib = self.velocity._lib
        self.device = self.velocity.device
        self.N = self.velocity.N
        self.n_v, self.n_p = self.velocity.n, self.pressure.n
        self.tau = self.velocity.tau
        indptr, indices, data = csr_arrays(B)
        if indptr.size != self.n_p + 1 or (indices.size and int(indices.max()) >= self.n_v):
            raise ValueError("B must be the n_p x n_v divergence matrix")
        self._s = C.c_void_p()
        self.velocity._check(self._lib.ctl_stokes_create(self.velocity._h, self.pressure._h, indptr.ctypes.data,
                                                         indices.ctypes.data, data.ctypes.data, C.byref(self._s)))
        if self._K_p_solver is not None:
            self.velocity._check(self._lib.ctl_stokes_set_laplacian_p(self._s, self._K_p_solver.ctypes.data))
        self._pc_ready = False

    def set_forward(self, K_v, D_p=None):
        """New forward matrices of a Picard iteration (control/control.py:5109-5118: every outer iteration
        re-linearises around the new velocity): velocity-space ``D_v_i`` and, when given, pressure-space
        ``D_p_i``.  The Laplacian of ``solver_K_p`` stays."""
        self.velocity.set_K(K_v)
        if D_p is not None:
            if self._K_p_solver is None:
                raise ValueError("construct the StokesSystem with D_p= to change the pressure-space forward matrices")
            self.pressure.set_K(D_p)
        self._pc_ready = False

    # ------------------------------------------------------------------ plumbing
    def _call(self, fn, *args):
        cur = torch.cuda.current_stream(self.device)
        self.velocity.stream.wait_stream(cur)
        rc = fn(self._s, *args)
        cur.wait_stream(self.velocity.stream)
        self.velocity._check(rc)

    def close(self):
        if getattr(self, "_s", None) is not None and self._s:
            self._lib.ctl_stokes_destroy(self._s)
            self._s = C.c_void_p()
        for name in ("pressure", "velocity"):
            sysm = getattr(self, name, None)
            if sysm is not None:
                sysm.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def vec_len(self):
        return int(self._lib.ctl_stokes_vec_len(self._s))

    def kernel_launches(self):
        return int(self._lib.ctl_kernel_launches(self.velocity._h)) + int(self._lib.ctl_kernel_launches(self.pressure._h))

    def to_device(self, x_0, x_1):
        host = np.concatenate([np.asarray(_as_host_f64(x_0), dtype=np.float64).ravel(),
                               np.asarray(_as_host_f64(x_1), dtype=np.float64).ravel()])
        if host.size != self.vec_len():
            raise ValueError(f"vector has {host.size} entries, expected {self.vec_len()}")
        return torch.from_numpy(host).to(self.device)

    def to_host_blocks(self, x_dev):
        a = x_dev.detach().cpu().numpy()
        L0 = 2 * self.N * self.n_v
        return a[:L0].reshape(2 * self.N, self.n_v), a[L0:].reshape(2 * self.N, self.n_p)

    def velocity_state_to_host(self, x_dev):
        """The N velocity-state blocks of an outer device vector (its first N n_v entries) as a host array of shape
        (N, n_v): all a Picard loop needs to assemble ``D_v_i`` / ``D_p_i`` at the iterate."""
        self._check_vec(x_dev, "velocity_state_to_host")
        return x_dev[:self.N * self.n_v].cpu().numpy().reshape(self.N, self.n_v)

    def new_vector(self):
        """A zero outer device vector (block-major, ``vec_len()`` entries)."""
        return torch.zeros(self.vec_len(), dtype=torch.float64, device=self.device)

    def _check_vec(self, t, what):
        if not isinstance(t, torch.Tensor) or t.numel() != self.vec_len() or t.dtype != torch.float64 \
                or not t.is_cuda or not t.is_contiguous():
            raise ValueError(f"{what} needs contiguous float64 CUDA vectors of vec_len() entries")

    # ------------------------------------------------------------------ operator / preconditioner
    def apply(self, x_dev, y_dev=None):
        """y = A x (MultiBlockSystemMatrix.mult, preconditioner/preconditioner.py:375-543)."""
        if y_dev is None:
            y_dev = torch.empty_like(x_dev)
        self._call(self._lib.ctl_stokes_apply, x_dev.data_ptr(), y_dev.data_ptr())
        return y_dev

    def setup_preconditioner(self, *, lambda_v_bounds=None, lambda_p_bounds=None, inner_its=5, mass_p_steps=20,
                             amg=None, amg_p=None, Multigrid=False):
        """The in-built pressure-Schur preconditioner (control/control.py:4299-4687).  ``amg`` /
        ``amg_p``: parameters of the AMG stand-in for the velocity sweeps / the K_p solves."""
        o = L.ctl_stokes_pc_options()
        self.velocity._check(self._lib.ctl_stokes_pc_default_options(C.byref(o)))
        if Multigrid:                                   # construct_pc(Multigrid, ...), control/control.py:1954-1965
            o.velocity.solver_0 = L.CTL_S0_AMG
        elif lambda_v_bounds is not None:
            o.velocity.solver_0 = L.CTL_S0_CHEBYSHEV
            o.velocity.cheb_emin, o.velocity.cheb_emax = float(lambda_v_bounds[0]), float(lambda_v_bounds[1])
        if lambda_p_bounds is not None:
            o.mass_p = L.CTL_S0_CHEBYSHEV
            o.lambda_p_min, o.lambda_p_max = float(lambda_p_bounds[0]), float(lambda_p_bounds[1])
        o.inner_its = int(inner_its)
        o.mass_p_steps = int(mass_p_steps)
        names = (("cycles", "cycles"), ("nu", "nu"), ("max_levels", "max_levels"), ("coarse_max", "coarse_max"),
                 ("theta", "theta"), ("lo", "lo"), ("hi", "hi"))
        amg = dict(amg or {})
        for key, field in names + (("nu_fine", "nu_fine"), ("acc_lo", "acc_lo"), ("acc_hi", "acc_hi")):
            if key in amg:
                setattr(o.velocity, "amg_" + field, amg.pop(key))
        amg_p = dict(amg_p or {})
        for key, field in names:
            if key in amg_p:
                setattr(o, "amg_p_" + field, amg_p.pop(key))
        if amg or amg_p:
            raise TypeError(f"unknown AMG options {sorted(amg) + sorted(amg_p)}")
        self._call(self._lib.ctl_stokes_pc_setup, C.byref(o))
        self._pc_ready = True

    def pc_apply(self, b_dev, u_dev=None, raw=False):
        """``Preconditioner.apply`` (raw=False) or the bare ``pc_fn`` (raw=True)."""
        if u_dev is None:
            u_dev = torch.zeros_like(b_dev)
        fn = self._lib.ctl_stokes_pc_fn if raw else self._lib.ctl_stokes_pc_apply
        self._call(fn, b_dev.data_ptr(), u_dev.data_ptr())
        return u_dev

    def lift_bc_device(self, g, b_dev):
        """Lift inhomogeneous velocity Dirichlet data into the outer device right-hand side ``b_dev`` (block-major,
        ``vec_len()`` entries) in place (``ctl_stokes_lift_bc``): velocity rows as ``MultiBlockSystem.lift_bc_device``,
        divergence rows ``b_1_0 -= tau B g`` then T_2 for CN (control/control.py:4107-4119, 4207-4219).  ``g``:
        (n_t, len(bc_dofs_v)) host array or CUDA tensor.  Returns ``b_dev``."""
        if b_dev.numel() != self.vec_len() or b_dev.dtype != torch.float64 or not b_dev.is_cuda \
                or not b_dev.is_contiguous():
            raise ValueError("lift_bc_device needs a contiguous float64 CUDA vector of vec_len() entries")
        g_dev = self.velocity._bc_values_device(g)
        self._call(self._lib.ctl_stokes_lift_bc, g_dev.data_ptr(), b_dev.data_ptr())
        return b_dev

    def nonlinear_residual(self, b_dev, x_dev, r_dev):
        """Residual of the Navier-Stokes Picard loop on outer device vectors (``ctl_stokes_nonlinear_residual``;
        replaces ``res_eval`` of control/control.py:4979-5072): fills ``r_dev = b - A_raw x`` -- the right-hand side
        of the increment solve, constrained velocity rows zero -- and returns the norm the reference's loop tests,
        that of the untransformed parts (r00, r01, r10, r11).  ``A_raw`` is the outer operator with ``D_v`` at the
        iterate (call ``set_forward`` first) and the RAW coupling products: unlike ``apply`` it does not centre the
        pressure parts, because the reference's residual does not."""
        for t in (b_dev, x_dev, r_dev):
            self._check_vec(t, "nonlinear_residual")
        out = C.c_double()
        self._call(self._lib.ctl_stokes_nonlinear_residual, b_dev.data_ptr(), x_dev.data_ptr(), r_dev.data_ptr(),
                   C.byref(out))
        return float(out.value)

    def time_divergence_products(self, reps=20):
        """Average milliseconds and algorithmic bytes of the batched ``tau B X`` / ``Y += tau B^T X``
        panel products (``ctl_stokes_time``)."""
        out = (C.c_double * 4)()
        self._call(self._lib.ctl_stokes_time, int(reps), out)
        return {"B_ms": out[0], "B_bytes": out[1], "BT_ms": out[2], "BT_bytes": out[3]}

    # ------------------------------------------------------------------ solve
    def solve_device(self, b_dev, u_dev, *, solver_parameters=None, pc="builtin"):
        if solver_parameters is None:                             # control/control.py:4291-4297
            solver_parameters = {"linear_solver": "fgmres", "maximum_iterations": 100,
                                 "relative_tolerance": 1.0e-6, "absolute_tolerance": 0.0}
        kind = {"none": L.CTL_PC_NONE, "builtin": L.CTL_PC_BUILTIN, "callback": L.CTL_PC_CALLBACK}[pc]
        if kind == L.CTL_PC_BUILTIN and not self._pc_ready:
            raise L.CtlError("call setup_preconditioner() first")
        o = self.velocity._krylov_options(solver_parameters, kind)
        res = L.ctl_solve_result()
        self._call(self._lib.ctl_stokes_solve, b_dev.data_ptr(), u_dev.data_ptr(), C.byref(o), C.byref(res))
        return KSPInfo(res)

    def _install_callback(self, pc_fn):
        """``P=`` of ``incompressible_linear_solve``: ``pc_fn(u_0, u_1, b_0, b_1)`` on host block arrays of shape
        (2N, n_v) and (2N, n_p); ``b_*`` projected and read-only, ``u_*`` zero, filled in place
        (preconditioner/preconditioner.py:620-627)."""
        from .system import _error_flag, _wrap_device_ptr
        sys_ = self

        def trampoline(_user, b_ptr, u_ptr):
            try:
                b = _wrap_device_ptr(b_ptr, sys_.vec_len(), sys_.device)
                u = _wrap_device_ptr(u_ptr, sys_.vec_len(), sys_.device)
                b0, b1 = sys_.to_host_blocks(b)
                u0, u1 = np.zeros_like(b0), np.zeros_like(b1)
                pc_fn(u0, u1, b0, b1)
                u.copy_(sys_.to_device(u0, u1))
                torch.cuda.current_stream(sys_.device).synchronize()
                return 0
            except Exception:                                     # flag_errors, preconditioner.py:64-72
                _error_flag[0] = True
                import traceback
                traceback.print_exc()
                return 1
        cb = L.PC_CALLBACK(trampoline)
        self._cb_keepalive = cb
        self.velocity._check(self._lib.ctl_stokes_set_pc_callback(self._s, cb, None))

    def builtin_pc_fn(self):
        """The in-built pressure-Schur preconditioner as a ``P``-compatible callable on host block arrays."""
        def pc_fn(u_0, u_1, b_0, b_1):
            u = torch.empty(self.vec_len(), dtype=torch.float64, device=self.device)
            self._call(self._lib.ctl_stokes_pc_fn, self.to_device(b_0, b_1).data_ptr(), u.data_ptr())
            r0, r1 = self.to_host_blocks(u)
            np.copyto(_as_host_f64(u_0).reshape(r0.shape), r0)
            np.copyto(_as_host_f64(u_1).reshape(r1.shape), r1)
        return pc_fn

    def solve(self, u_0, u_1, b_0, b_1, *, solver_parameters=None, pc_fn="builtin"):
        """``MultiBlockSystem.solve`` of the outer system on host block arrays: ``u_0`` (2N, n_v)
        and ``u_1`` (2N, n_p) carry the initial guess in and the solution out."""
        pc = "none" if pc_fn is None else pc_fn
        if callable(pc_fn):                     # a user P(u_0, u_1, b_0, b_1): control/control.py:4686-4689
            self._install_callback(pc_fn)
            pc = "callback"
        elif pc not in ("none", "builtin"):
            raise ValueError("the Stokes system takes pc_fn=None, 'builtin' or a callable P(u_0, u_1, b_0, b_1)")
        b = self.to_device(b_0, b_1)
        u = self.to_device(u_0, u_1)
        info = self.solve_device(b, u, solver_parameters=solver_parameters, pc=pc)
        r0, r1 = self.to_host_blocks(u)
        np.copyto(_as_host_f64(u_0).reshape(r0.shape), r0)
        np.copyto(_as_host_f64(u_1).reshape(r1.shape), r1)
        sp = solver_parameters or {}
        if not sp.get("preconditioner", False) and info.reason <= 0:   # preconditioner.py:756, 768-770
            raise RuntimeError("Solver failed to converge")
        return info
