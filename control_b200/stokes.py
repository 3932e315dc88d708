"""Host-side mirror of the outer block system of instationary Stokes control.

``StokesSystem`` plays the role of the ``MultiBlockSystem`` the reference builds in
``Control.Instationary.incompressible_linear_solve`` (control/control.py:3592-4725, system
construction at 4273-4289): block_00 = the heat-type KKT system on the velocity space,
block_01 / block_10 = diag(tau B^T) / diag(tau B), block_11 = None, with sub-block T
transforms (preconditioner/preconditioner.py:471-525), DirichletBCNullspace on the velocity
blocks and ConstantNullspace on the pressure blocks.  It is constructed from the five
spatial matrices the blocks are made of; every numeric operation runs in libctl_b200.so.

Vectors at this boundary are block-major: ``x_0`` of shape (2N, n_v) = [v | zeta] and ``x_1``
of shape (2N, n_p) = [mu | p], or one flat device vector [x_0 | x_1].  On several ranks (``world > 1``)
each rank holds its own rows of both spaces, PETSc's split of each (``velocity_rows``,
``pressure_rows``): ``x_0`` of shape (2N, n_v_local), ``x_1`` of shape (2N, n_p_local).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L
from .system import MultiBlockSystem, _DeviceSystem, csr_arrays, fgmres_defaults

__all__ = ["StokesSystem"]


class StokesSystem(_DeviceSystem):
    _SET_CALLBACK = "ctl_stokes_set_pc_callback"

    def __init__(self, M_v, K_v, B, M_p, K_p, *, n_t, beta, CN, time_interval=(0.0, 1.0), bc_dofs_v=(),
                 epsilon=1e-3, device=None, D_p=None, velocity_block_size=1, rank=0, world=1):
        """``K_v``: the forward matrix on the velocity space (one matrix or n_t matrices ``D_v_i``).  ``K_p``: the
        pressure Laplacian ``solver_K_p`` inverts (control/control.py:3746, 4300-4309).  ``D_p``: the forward
        form on the PRESSURE space (``D_p_i``, control/control.py:3787-3789; one matrix or n_t matrices) of the
        pressure-space KKT multiply; default ``K_p`` (the Stokes forward operator).  ``velocity_block_size``: block
        size of the velocity space (2 for a 2-D ``VectorFunctionSpace``): the velocity sweeps then run on the scalar
        block of ``I_2 (x) S`` (``MultiBlockSystem(block_size=)``); one GPU only.  ``rank`` / ``world``: this
        process's rank of ``world`` (one GPU each); with ``world > 1`` call ``init_comm`` before anything else."""
        if int(velocity_block_size) > 1 and world > 1:
            raise ValueError("velocity_block_size > 1 runs on one GPU: block-scalar sweeps are not available with "
                             "world > 1")
        self.velocity = MultiBlockSystem(M_v, K_v, n_t=n_t, beta=beta, CN=CN, time_interval=time_interval,
                                         bc_dofs=bc_dofs_v, epsilon=epsilon, device=device,
                                         block_size=velocity_block_size, rank=rank, world=world)
        self.pressure = MultiBlockSystem(M_p, K_p if D_p is None else D_p, n_t=n_t, beta=beta, CN=CN,
                                         time_interval=time_interval, bc_dofs=(), epsilon=epsilon,
                                         device=self.velocity.device.index, stream=self.velocity.stream,
                                         rank=rank, world=world)
        self.rank, self.world = rank, world
        self._K_p_solver = None if D_p is None else np.ascontiguousarray(self.pressure._same_pattern(K_p))
        self._lib = self.velocity._lib
        self.device = self.velocity.device
        self._stream = self.velocity.stream
        self.N = self.velocity.N
        self.n_v, self.n_p = self.velocity.n, self.pressure.n
        self.n_v_local, self.n_p_local = self.velocity.n_local, self.pressure.n_local
        self.velocity_rows = slice(self.velocity.row_begin, self.velocity.row_begin + self.n_v_local)
        self.pressure_rows = slice(self.pressure.row_begin, self.pressure.row_begin + self.n_p_local)
        self.tau = self.velocity.tau
        indptr, indices, data = csr_arrays(B)
        if indptr.size != self.n_p + 1 or (indices.size and int(indices.max()) >= self.n_v):
            raise ValueError("B must be the n_p x n_v divergence matrix")
        self._B = (indptr, indices, data)
        self._s = C.c_void_p()
        self._pc_ready = False
        if world == 1:
            self._create()

    def _create(self):
        indptr, indices, data = self._B
        self._check(self._lib.ctl_stokes_create(self.velocity._h, self.pressure._h, indptr.ctypes.data,
                                                indices.ctypes.data, data.ctypes.data, C.byref(self._s)))
        if self._K_p_solver is not None:
            self._check(self._lib.ctl_stokes_set_laplacian_p(self._s, self._K_p_solver.ctypes.data))

    def init_comm(self, dist=None):
        """Several ranks: the NCCL communicators of both spaces (``MultiBlockSystem.init_comm``), then the outer
        system, whose divergence products exchange rows through them.  Every rank passes the global matrices."""
        if self.world == 1:
            return
        self.velocity.init_comm(dist)
        self.pressure.init_comm(dist)
        self._create()

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
    @property
    def _handle(self):
        return self._s

    def _check(self, rc):
        self.velocity._check(rc)            # the library records the Stokes system's errors on the velocity handle

    def close(self):
        """Release the outer system and both handles; collective with world > 1 (see ``MultiBlockSystem.close``)."""
        if getattr(self, "_s", None) is not None and self._s:
            self._lib.ctl_stokes_destroy(self._s)
            self._s = C.c_void_p()
        for name in ("pressure", "velocity"):
            sysm = getattr(self, name, None)
            if sysm is not None:
                sysm.close()

    def vec_len(self, layout=L.CTL_LAYOUT_BLOCK_MAJOR):
        if layout != L.CTL_LAYOUT_BLOCK_MAJOR:
            raise ValueError("the outer vectors of the Stokes system are block-major")
        return int(self._lib.ctl_stokes_vec_len(self._s))

    def kernel_launches(self):
        return int(self._lib.ctl_kernel_launches(self.velocity._h)) + int(self._lib.ctl_kernel_launches(self.pressure._h))

    def to_host_blocks(self, x_dev):
        a = x_dev.detach().cpu().numpy()
        L0 = 2 * self.N * self.n_v_local
        return a[:L0].reshape(2 * self.N, self.n_v_local), a[L0:].reshape(2 * self.N, self.n_p_local)

    def allgather_blocks(self, x_0, x_1):
        """This rank's block arrays (2N, n_v_local), (2N, n_p_local) -> the global (2N, n_v), (2N, n_p) on every
        rank."""
        return self.velocity.allgather_blocks(x_0), self.pressure.allgather_blocks(x_1)

    def velocity_state_to_host(self, x_dev):
        """The N velocity-state blocks of an outer device vector (its first N n_v_local entries) as a host array of
        shape (N, n_v_local): all a Picard loop needs to assemble ``D_v_i`` / ``D_p_i`` at the iterate."""
        self._check_vecs("velocity_state_to_host", x_dev)
        return x_dev[:self.N * self.n_v_local].cpu().numpy().reshape(self.N, self.n_v_local)

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
        self._check(self._lib.ctl_stokes_pc_default_options(C.byref(o)))
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
        self._check_vecs("lift_bc_device", b_dev)
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
        self._check_vecs("nonlinear_residual", b_dev, x_dev, r_dev)
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
            solver_parameters = fgmres_defaults(False)
        return self._ksp(self._lib.ctl_stokes_solve, b_dev, u_dev, solver_parameters, pc)

    builtin_pc_fn = _DeviceSystem.pc_fn         # the in-built pressure-Schur preconditioner as a host ``P``

    def solve(self, u_0, u_1, b_0, b_1, *, solver_parameters=None, pc_fn="builtin"):
        """``MultiBlockSystem.solve`` of the outer system on host block arrays ``u_0`` (2N, n_v) and ``u_1`` (2N, n_p),
        with the in-built preconditioner by default."""
        return super().solve(u_0, u_1, b_0, b_1, solver_parameters=solver_parameters, pc_fn=pc_fn)
