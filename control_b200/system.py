"""Host-side mirror of the reference's block-system layer for the instationary KKT path.

``MultiBlockSystem`` keeps the role and the call shapes of the reference class
(preconditioner/preconditioner.py:216-786) -- ``solve(u_0, u_1, b_0, b_1, *,
solver_parameters, pc_fn)``, a shell-matrix context with ``mult(A, x, y)`` and a shell-PC
context with ``apply(pc, x, y)`` -- but is constructed from the two or three distinct
spatial matrices the 8N-4 UFL blocks are made of (control/control.py:2889-2978) instead
of the dict of forms, because only those matrices ever cross into the CUDA library.
Every numeric operation is executed by libctl_b200.so; PyTorch only owns device buffers.

Vectors at this boundary are block-major like the reference's mixed PETSc vectors:
arrays of shape (N, n) per block row, or flat arrays of 2*N*n.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L

__all__ = ["MultiBlockSystem", "KSPInfo", "csr_arrays", "finish_ksp", "gmres_defaults", "fgmres_defaults"]

_KSP_TYPES = {"gmres": L.CTL_KSP_GMRES, "fgmres": L.CTL_KSP_FGMRES, "minres": L.CTL_KSP_MINRES}

# module-global error flag of the reference (preconditioner/preconditioner.py:29, 64-72,
# 771-772).  Unlike the reference it is reset at the start of every solve.
_error_flag = [False]


def csr_arrays(A):
    """(indptr int32, indices int32, data float64) of a scipy CSR matrix or a triple.
    A petsc4py ``Mat`` can be passed as ``A.getValuesCSR()``."""
    if isinstance(A, (tuple, list)) and len(A) == 3:
        indptr, indices, data = A
    else:
        A = A.tocsr()
        if not A.has_sorted_indices:
            A = A.sorted_indices()
        indptr, indices, data = A.indptr, A.indices, A.data
    return (np.ascontiguousarray(indptr, dtype=np.int32),
            np.ascontiguousarray(indices, dtype=np.int32),
            np.ascontiguousarray(data, dtype=np.float64))


class KSPInfo:
    """What the reference gets back from ``MultiBlockSystem.solve`` (the PETSc KSP,
    preconditioner/preconditioner.py:786), reduced to the queries its callers make."""

    def __init__(self, res):
        self.its = int(res.its)
        self.reason = int(res.reason)
        self.n_mult = int(res.n_mult)
        self.n_pc = int(res.n_pc)
        self.rnorm = float(res.rnorm)
        self.ref_norm = float(res.ref_norm)
        self.history = [float(res.history[i]) for i in range(min(res.n_history, L.CTL_HISTORY_MAX))]
        self.seconds_total = float(res.seconds_total)
        self.seconds_mult = float(res.seconds_mult)
        self.seconds_pc = float(res.seconds_pc)

    def getConvergedReason(self):
        return self.reason

    def getIterationNumber(self):
        return self.its

    def getResidualNorm(self):
        return self.rnorm


def _as_host_f64(x):
    """numpy view of a numpy array, a CPU torch tensor or a PETSc Vec."""
    if isinstance(x, np.ndarray):
        return x
    if isinstance(x, torch.Tensor):
        return x.detach().cpu().numpy()
    if hasattr(x, "getArray"):                       # petsc4py.PETSc.Vec
        return x.getArray(readonly=False)
    return np.asarray(x)


def gmres_defaults(monitor):
    """The heat-type drivers' ``solver_parameters`` when the caller gives none (control/control.py:562-568,
    3260-3266)."""
    return {"linear_solver": "gmres", "gmres_restart": 10, "maximum_iterations": 50, "relative_tolerance": 1.0e-6,
            "absolute_tolerance": 0.0, "monitor_convergence": monitor}


def fgmres_defaults(monitor, max_it=100):
    """The Stokes-type drivers' ``solver_parameters`` when the caller gives none: ``max_it`` 100 for the instationary
    ones (control/control.py:4291-4297), 50 for the stationary one (1088-1094)."""
    return {"linear_solver": "fgmres", "fgmres_restart": 10, "maximum_iterations": max_it,
            "relative_tolerance": 1.0e-6, "absolute_tolerance": 0.0, "monitor_convergence": monitor}


def finish_ksp(info, solver_parameters):
    """The end of the reference's ``MultiBlockSystem.solve`` (preconditioner/preconditioner.py:749-770): print the
    residual history when ``monitor_convergence`` is set (the reference's default is True), and raise when the solve
    did not converge unless ``preconditioner`` is set."""
    if solver_parameters.get("monitor_convergence", True):
        for it, r_norm in enumerate(info.history):
            print(f"KSP: iteration {it:d}, residual norm {r_norm:.16e}")
    if not solver_parameters.get("preconditioner", False) and info.reason <= 0:
        raise RuntimeError("Solver failed to converge")


class _DeviceSystem:
    """What the heat-type and the Stokes systems share at the host boundary: ordered library calls, block-major
    device vectors, the Krylov options and the host ``solve`` with the reference's ``pc_fn`` hook.  A subclass
    supplies ``_lib``, ``device``, ``_stream``, ``_pc_ready``, its handle (``_handle``, ``_check``), ``vec_len``,
    ``to_host_blocks``, ``pc_apply``, ``solve_device`` and the name of its callback setter (``_SET_CALLBACK``)."""

    @property
    def stream(self):
        """The CUDA stream the library launches on (time it with events recorded here)."""
        return self._stream

    def _call(self, fn, *args):
        """Library call ordered after the work already queued on torch's current stream,
        and torch's later work ordered after the call."""
        cur = torch.cuda.current_stream(self.device)
        self._stream.wait_stream(cur)
        rc = fn(self._handle, *args)
        cur.wait_stream(self._stream)
        self._check(rc)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ device vectors
    def new_vector(self, layout=L.CTL_LAYOUT_BLOCK_MAJOR):
        """A zero device vector of ``vec_len(layout)`` entries."""
        return torch.zeros(self.vec_len(layout), dtype=torch.float64, device=self.device)

    def to_device(self, x_0, x_1=None):
        """Block-major device vector from the two host block arrays of ``to_host_blocks`` or a flat array."""
        if x_1 is None:
            host = np.ascontiguousarray(_as_host_f64(x_0), dtype=np.float64).ravel()
        else:
            host = np.concatenate([np.asarray(_as_host_f64(x_0), dtype=np.float64).ravel(),
                                   np.asarray(_as_host_f64(x_1), dtype=np.float64).ravel()])
        if host.size != self.vec_len():
            raise ValueError(f"vector has {host.size} entries, expected {self.vec_len()}")
        return torch.from_numpy(host).to(self.device)

    def _to_host_arrays(self, x_dev, x_0, x_1):
        """Copy a block-major device vector into the caller's host block arrays in place."""
        r0, r1 = self.to_host_blocks(x_dev)
        np.copyto(_as_host_f64(x_0).reshape(r0.shape), r0)
        np.copyto(_as_host_f64(x_1).reshape(r1.shape), r1)

    def _check_vecs(self, what, *ts, count=None, layout=L.CTL_LAYOUT_BLOCK_MAJOR):
        """Device vector arguments: contiguous float64 CUDA tensors of ``count`` (default ``vec_len(layout)``)
        entries."""
        n = self.vec_len(layout) if count is None else count
        for t in ts:
            if not isinstance(t, torch.Tensor) or t.numel() != n or t.dtype != torch.float64 or not t.is_cuda \
                    or not t.is_contiguous():
                raise ValueError(f"{what} needs contiguous float64 CUDA tensors of {n} entries")

    # ------------------------------------------------------------------ solve
    def _pc_kind(self, pc):
        kind = {"none": L.CTL_PC_NONE, "builtin": L.CTL_PC_BUILTIN, "callback": L.CTL_PC_CALLBACK}[pc]
        if kind == L.CTL_PC_BUILTIN and not self._pc_ready:
            raise L.CtlError("call setup_preconditioner() first")
        return kind

    def _krylov_options(self, solver_parameters, pc):
        kind = self._pc_kind(pc)
        sp = solver_parameters or {}
        o = L.ctl_krylov_options()
        self._check(self._lib.ctl_krylov_default_options(C.byref(o)))
        ksp_type = sp.get("linear_solver", "fgmres")              # preconditioner.py:733
        if ksp_type not in _KSP_TYPES:
            raise ValueError(f"unsupported linear_solver {ksp_type!r}")
        o.ksp_type = _KSP_TYPES[ksp_type]
        o.rtol = float(sp["relative_tolerance"])                  # required keys: 739-740
        o.atol = float(sp["absolute_tolerance"])
        if sp.get("divergence limit") is not None:
            o.divtol = float(sp["divergence limit"])
        o.max_it = int(sp.get("maximum_iterations", 1000))
        if "gmres_restart" in sp:                                 # "fgmres_restart" is never read: 747-748
            o.restart = int(sp["gmres_restart"])
        # "pc_side" (735-736) and "norm_type" (744-746) are forwarded to PETSc by the reference.  krylov.cuh
        # implements PETSc's defaults for each solver -- left + preconditioned norm for gmres / minres, right +
        # unpreconditioned norm for fgmres -- so any other request is refused instead of silently ignored (a
        # different side or norm changes the convergence test and the iteration count)
        right = ksp_type == "fgmres"
        side = sp.get("pc_side")
        if side is not None and str(side).lower() not in (("right", "2", "pc_right") if right else ("left", "1", "pc_left")):
            raise ValueError(f"pc_side={side!r} is not implemented for {ksp_type}: only PETSc's default side "
                             f"({'right' if right else 'left'})")
        norm = sp.get("norm_type")
        if norm is not None and str(norm).lower() not in (
                ("default", "-1", "unpreconditioned", "2", "norm_unpreconditioned") if right
                else ("default", "-1", "preconditioned", "1", "norm_preconditioned")):
            raise ValueError(f"norm_type={norm!r} is not implemented for {ksp_type}: only PETSc's default "
                             f"({'unpreconditioned' if right else 'preconditioned'})")
        o.pc = kind
        return o

    def _ksp(self, entry, b_dev, u_dev, solver_parameters, pc, *args):
        """One Krylov solve through the C entry point ``entry(handle, b, u, *args, options, result)``."""
        o = self._krylov_options(solver_parameters, pc)
        res = L.ctl_solve_result()
        self._call(entry, b_dev.data_ptr(), u_dev.data_ptr(), *args, C.byref(o), C.byref(res))
        return KSPInfo(res)

    def pc_fn(self):
        """The in-built preconditioner as a ``P``-compatible callable ``pc_fn(u_0, u_1, b_0, b_1)`` on host block
        arrays (control/control.py:3245-3258, 4686-4689)."""
        def pc_fn(u_0, u_1, b_0, b_1):
            self._to_host_arrays(self.pc_apply(self.to_device(b_0, b_1), raw=True), u_0, u_1)
        return pc_fn

    def _install_callback(self, pc_fn):
        sys_ = self

        def trampoline(_user, b_ptr, u_ptr):
            try:
                b = _wrap_device_ptr(b_ptr, sys_.vec_len(), sys_.device)
                u = _wrap_device_ptr(u_ptr, sys_.vec_len(), sys_.device)
                # the library synchronised its stream before calling back
                b0, b1 = sys_.to_host_blocks(b)
                u0 = np.zeros_like(b0)
                u1 = np.zeros_like(b1)
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
        self._check(getattr(self._lib, self._SET_CALLBACK)(self._handle, cb, None))

    def solve(self, u_0, u_1, b_0, b_1, *, solver_parameters=None, pc_fn=None):
        """``MultiBlockSystem.solve`` (preconditioner/preconditioner.py:337-786) on the host block arrays of
        ``to_host_blocks``: u_* carry the initial guess in and the solution out.

        ``pc_fn``: None = identity (342-345); the string "builtin" = the in-built preconditioner running on the
        device (set up with ``setup_preconditioner``); a callable ``pc_fn(u_0, u_1, b_0, b_1)`` = the reference's
        user hook, called back every iteration on host block arrays: ``b_*`` projected and read-only, ``u_*`` zero,
        filled in place (620-627)."""
        _error_flag[0] = False
        if pc_fn is None:
            pc = "none"
        elif isinstance(pc_fn, str) and pc_fn == "builtin":
            pc = "builtin"
        elif callable(pc_fn):
            self._install_callback(pc_fn)
            pc = "callback"
        else:
            raise ValueError(f"pc_fn must be None, 'builtin' or a callable P(u_0, u_1, b_0, b_1), not {pc_fn!r}")
        b = self.to_device(b_0, b_1)
        u = self.to_device(u_0, u_1)
        info = self.solve_device(b, u, solver_parameters=solver_parameters, pc=pc)
        self._to_host_arrays(u, u_0, u_1)
        finish_ksp(info, solver_parameters or {})
        if _error_flag[0]:                                        # 771-772
            raise RuntimeError("Error encountered in PETSc solve")
        return info


class MultiBlockSystem(_DeviceSystem):
    _SET_CALLBACK = "ctl_set_pc_callback"

    def __init__(self, M, K, *, n_t, beta, CN, time_interval=(0.0, 1.0), bc_dofs=(),
                 epsilon=1e-3, device=None, rank=0, world=1, stream=None, block_size=1):
        """``block_size``: PETSc's Mat block size of the space (``M.petscmat.getBlockSize()``), dofs interleaved as
        ``bs * node + comp``.  With 2 or 3, the preconditioner runs its time sweeps on the scalar block ``S`` of
        matrices ``I_bs (x) S`` (``ctl_set_block_size``; ``pc_block_size`` tells whether they had that structure)."""
        block_size = int(block_size)
        if block_size not in (1, 2, 3):
            raise ValueError(f"block_size must be 1, 2 or 3, not {block_size}")
        if block_size > 1 and world > 1:
            raise ValueError("block_size > 1 runs on one GPU: block-scalar sweeps are not available with world > 1")
        self._lib = L.load()
        self._h = C.c_void_p()
        if not torch.cuda.is_available():
            raise L.CtlError("control_b200 needs a CUDA device (there is no CPU fallback)")
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        torch.cuda.set_device(self.device)
        indptr, indices, m_data = csr_arrays(M)
        self.n = int(indptr.size - 1)
        self.n_t = int(n_t)
        self.CN = bool(CN)
        self.beta = float(beta)
        t_0, T_f = time_interval
        self.tau = (T_f - t_0) / (n_t - 1.0)                 # control/control.py:2831
        # the library runs on its own stream (the legacy default stream cannot be captured
        # into the sweep CUDA graph); every call is fenced against torch's current stream
        self._stream = torch.cuda.Stream(self.device) if stream is None else stream
        cfg = L.ctl_config(n=self.n, n_t=self.n_t, CN=int(self.CN), device=self.device.index,
                           tau=self.tau, beta=self.beta, epsilon=float(epsilon),
                           stream=C.c_void_p(self._stream.cuda_stream), rank=rank, world=world)
        rc = self._lib.ctl_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            raise L.CtlError(f"ctl_create failed ({rc}): {self._lib.ctl_last_error(None).decode()}")
        self.N = int(self._lib.ctl_n_blocks(self._h))
        self.ld = int(self._lib.ctl_ld(self._h))
        self.n_local = int(self._lib.ctl_n_local(self._h))
        self.row_begin = int(self._lib.ctl_row_begin(self._h))
        self.rank, self.world = rank, world
        self._pattern = (indptr, indices)
        self._check(self._lib.ctl_set_pattern(self._h, indptr.ctypes.data, indices.ctypes.data,
                                              C.c_int64(indices.size)))
        self._check(self._lib.ctl_set_values(self._h, L.CTL_MAT_M, -1, m_data.ctypes.data))
        self.bc_dofs = np.ascontiguousarray(bc_dofs, dtype=np.int32)
        self._check(self._lib.ctl_set_bc(self._h, self.bc_dofs.ctypes.data, self.bc_dofs.size))
        self.block_size = block_size
        if block_size != 1:
            self._check(self._lib.ctl_set_block_size(self._h, block_size))
        self._pc_ready = False
        self._cb_keepalive = None
        self.set_K(K)

    # ------------------------------------------------------------------ plumbing
    @property
    def _handle(self):
        return self._h

    def _check(self, rc):
        L.check(self._h, rc)

    def close(self):
        """Release the handle.  With world > 1 this is collective (ctl_destroy): call it on every rank at the same
        point rather than leaving it to garbage collection, whose timing differs between processes."""
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.ctl_destroy(self._h)
            self._h = C.c_void_p()

    def _same_pattern(self, A):
        indptr, indices, data = csr_arrays(A)
        if indptr.size != self._pattern[0].size or indices.size != self._pattern[1].size or \
                not (np.array_equal(indptr, self._pattern[0]) and np.array_equal(indices, self._pattern[1])):
            raise ValueError("M and K must share one sparsity pattern (keep structural zeros)")
        return data

    def set_K(self, K, K_T=None):
        """Hand over the forward operator: one matrix (time independent) or a sequence of
        n_t matrices ``D_v_i`` (control/control.py:1887-1896, 2903-2904).  Called again by
        the Picard / Gauss-Newton loop with new values (control/control.py:3468-3504)."""
        if isinstance(K, (list, tuple)) and not (len(K) == 3 and isinstance(K[0], np.ndarray)):
            if len(K) != self.n_t:
                raise ValueError("need one K per time level")
            for i, Ki in enumerate(K):
                self._check(self._lib.ctl_set_values(self._h, L.CTL_MAT_K, i,
                                                     self._same_pattern(Ki).ctypes.data))
            if K_T is not None:
                for i, Ki in enumerate(K_T):
                    self._check(self._lib.ctl_set_values(self._h, L.CTL_MAT_KT, i,
                                                         self._same_pattern(Ki).ctypes.data))
        else:
            self._check(self._lib.ctl_set_values(self._h, L.CTL_MAT_K, -1,
                                                 self._same_pattern(K).ctypes.data))
            if K_T is not None:
                self._check(self._lib.ctl_set_values(self._h, L.CTL_MAT_KT, -1,
                                                     self._same_pattern(K_T).ctypes.data))
        self._check(self._lib.ctl_assemble(self._h))
        self._pc_ready = False

    def init_comm(self, dist=None):
        """Create the library's NCCL communicator: rank 0 draws the unique id, torch.distributed
        carries it to the other ranks (the one piece of plumbing done outside the library)."""
        if self.world == 1:
            return
        if dist is None:
            import torch.distributed as dist
        idbuf = (C.c_ubyte * 128)()
        if self.rank == 0:
            rc = self._lib.ctl_comm_unique_id(idbuf)
            if rc != 0:
                raise L.CtlError(f"ctl_comm_unique_id failed ({rc})")
        on_gpu = dist.get_backend() == "nccl"
        t = torch.tensor(list(idbuf), dtype=torch.uint8, device=self.device if on_gpu else "cpu")
        dist.broadcast(t, 0)
        raw = bytes(t.cpu().tolist())
        self._call(self._lib.ctl_comm_init, raw)

    # ------------------------------------------------------------------ device vectors
    def vec_len(self, layout=L.CTL_LAYOUT_BLOCK_MAJOR):
        return int(self._lib.ctl_vec_len(self._h, layout))

    def to_host_blocks(self, x_dev):
        a = x_dev.detach().cpu().numpy()
        half = self.N * self.n_local
        return a[:half].reshape(self.N, self.n_local), a[half:].reshape(self.N, self.n_local)

    def allgather_blocks(self, x_loc):
        """(N, n_local) blocks of every rank -> global (N, n) on every rank."""
        if self.world == 1:
            return x_loc
        import torch.distributed as dist
        parts = [None] * self.world
        dist.all_gather_object(parts, np.ascontiguousarray(x_loc))
        return np.concatenate(parts, axis=1)

    def convert(self, x_dev, src_layout, dst_layout):
        out = self.new_vector(dst_layout)
        self._call(self._lib.ctl_convert_layout, x_dev.data_ptr(), src_layout, out.data_ptr(), dst_layout)
        return out

    # ------------------------------------------------------------------ operator
    def apply(self, x_dev, y_dev=None, layout=L.CTL_LAYOUT_BLOCK_MAJOR):
        """y = A x on device vectors."""
        if y_dev is None:
            y_dev = torch.empty_like(x_dev)
        self._call(self._lib.ctl_kkt_apply, x_dev.data_ptr(), y_dev.data_ptr(), layout)
        return y_dev

    def time_apply(self, x_tf, y_tf, reps):
        ms = C.c_float()
        self._call(self._lib.ctl_time_kkt_apply, x_tf.data_ptr(), y_tf.data_ptr(), reps, C.byref(ms))
        return float(ms.value)

    def matshell(self):
        """Context for ``PETSc.Mat().createPython(((n, N), (n, N)), ctx, comm)``
        (preconditioner/preconditioner.py:720-722)."""
        return _MatShell(self)

    def pcshell(self, pc_fn=None):
        """Context for ``PETSc.PC().createPython(ctx, comm)`` (preconditioner.py:724-730)."""
        return _PCShell(self, pc_fn)

    # ------------------------------------------------------------------ preconditioner
    def setup_preconditioner(self, *, lambda_v_bounds=None, Multigrid=False, mode="triangular",
                             cheb_steps=20, **amg):
        """``Instationary.construct_pc(Multigrid, lambda_v_bounds, ...)``
        (control/control.py:1943-1991) + the AMG stand-in's parameters."""
        o = L.ctl_pc_options()
        self._check(self._lib.ctl_pc_default_options(C.byref(o)))
        o.mode = {"triangular": L.CTL_PCMODE_TRIANGULAR, "diagonal": L.CTL_PCMODE_DIAGONAL}[mode]
        if Multigrid:
            o.solver_0 = L.CTL_S0_AMG
        elif lambda_v_bounds is not None:
            o.solver_0 = L.CTL_S0_CHEBYSHEV
            o.cheb_emin, o.cheb_emax = float(lambda_v_bounds[0]), float(lambda_v_bounds[1])
        else:
            o.solver_0 = L.CTL_S0_JACOBI
        o.cheb_steps = int(cheb_steps)
        for key, field in (("cycles", "amg_cycles"), ("nu", "amg_nu"), ("nu_fine", "amg_nu_fine"),
                           ("max_levels", "amg_max_levels"),
                           ("coarse_max", "amg_coarse_max"), ("theta", "amg_theta"),
                           ("lo", "amg_lo"), ("hi", "amg_hi"), ("acc_lo", "amg_acc_lo"),
                           ("acc_hi", "amg_acc_hi")):
            if key in amg:
                setattr(o, field, amg.pop(key))
        if amg:
            raise TypeError(f"unknown AMG options {sorted(amg)}")
        self._check(self._lib.ctl_pc_setup(self._h, C.byref(o)))
        self._pc_ready = True
        self._pc_opts = o

    @property
    def pc_block_size(self):
        """Block size the preconditioner's time sweeps run with: ``block_size`` when every sweep matrix is
        ``I_bs (x) S``, 1 when one is not (or ``block_size`` is 1); -1 before ``setup_preconditioner``."""
        return int(self._lib.ctl_pc_block_size(self._h))

    def pc_apply(self, b_dev, u_dev=None, layout=L.CTL_LAYOUT_BLOCK_MAJOR, raw=False):
        """``Preconditioner.apply`` (raw=False) or the bare ``pc_fn`` (raw=True)."""
        if u_dev is None:
            u_dev = torch.zeros_like(b_dev)
        fn = self._lib.ctl_pc_fn if raw else self._lib.ctl_pc_apply
        self._call(fn, b_dev.data_ptr(), u_dev.data_ptr(), layout)
        return u_dev

    # ------------------------------------------------------------------ solve
    def solve_device(self, b_dev, u_dev, *, solver_parameters, pc="builtin",
                     layout=L.CTL_LAYOUT_BLOCK_MAJOR):
        """KSP solve on device vectors; u_dev holds the initial guess and the solution."""
        return self._ksp(self._lib.ctl_solve, b_dev, u_dev, solver_parameters, pc, layout)

    def solve_host(self, u_host, b_host, *, solver_parameters, pc="builtin"):
        """``ctl_solve_host``: the end-to-end C entry point.  ``b_host`` / ``u_host`` are flat
        block-major float64 numpy arrays (``u_host``: initial guess in, solution out); the
        library copies them to the device and back itself."""
        o = self._krylov_options(solver_parameters, pc)
        if b_host.dtype != np.float64 or u_host.dtype != np.float64 or not b_host.flags.c_contiguous \
                or not u_host.flags.c_contiguous or b_host.size != self.vec_len() or u_host.size != self.vec_len():
            raise ValueError("solve_host needs contiguous float64 arrays of vec_len() entries")
        res = L.ctl_solve_result()
        self._call(self._lib.ctl_solve_host, b_host.ctypes.data, u_host.ctypes.data, C.byref(o), C.byref(res))
        return KSPInfo(res)

    def residual_norm(self, b_dev, x_dev, layout=L.CTL_LAYOUT_BLOCK_MAJOR):
        out = C.c_double()
        self._call(self._lib.ctl_kkt_residual_norm, b_dev.data_ptr(), x_dev.data_ptr(), layout, C.byref(out))
        return float(out.value)

    def nonlinear_residual(self, b_dev, x_dev, r_dev, layout=L.CTL_LAYOUT_BLOCK_MAJOR):
        """Residual of the outer Picard / Gauss-Newton loop on device vectors (``ctl_nonlinear_residual``; replaces
        ``non_linear_res_eval``, control/control.py:2442-2818): fills ``r_dev = b - A x`` (constrained rows zero) --
        the right-hand side of the increment solve -- and returns the norm of the untransformed residual, the
        quantity the reference's loop tests.  ``A`` carries ``D_v`` at the iterate: call ``set_K`` first."""
        out = C.c_double()
        self._call(self._lib.ctl_nonlinear_residual, b_dev.data_ptr(), x_dev.data_ptr(), r_dev.data_ptr(), layout,
                   C.byref(out))
        return float(out.value)

    def objective_device(self, v_dev, zeta_dev, v_hat_dev):
        """J_h from device arrays of n_t levels x n_local (level-major; this rank's rows), evaluated on the GPU;
        on several ranks every rank receives the global value."""
        self._check_vecs("objective_device", v_dev, zeta_dev, v_hat_dev, count=self.n_t * self.n_local)
        out = C.c_double()
        self._call(self._lib.ctl_objective, v_dev.data_ptr(), zeta_dev.data_ptr(), v_hat_dev.data_ptr(), C.byref(out))
        return float(out.value)

    def build_rhs_device(self, v_hat_dev, f_nodal_dev, v_0=None, bc_values=None):
        """Block-major device right-hand side of ``linear_solve`` from nodal data on the device
        (n_t levels x n_local each: this rank's rows); ``v_0``: host initial condition (all n entries) or None
        (``ctl_build_rhs``).  ``bc_values``: None (homogeneous Dirichlet data) or the (n_t, len(bc_dofs))
        boundary values of the state, lifted in with ``lift_bc_device``."""
        self._check_vecs("build_rhs_device", v_hat_dev, f_nodal_dev, count=self.n_t * self.n_local)
        if v_0 is not None and np.size(v_0) != self.n:
            raise ValueError("build_rhs_device: v_0 must hold all n entries")
        b = self.new_vector()
        v0 = None if v_0 is None else np.ascontiguousarray(v_0, dtype=np.float64)
        self._call(self._lib.ctl_build_rhs, v_hat_dev.data_ptr(), f_nodal_dev.data_ptr(),
                   None if v0 is None else v0.ctypes.data, b.data_ptr())
        if bc_values is not None:
            self.lift_bc_device(bc_values, b)
        return b

    def _bc_values_device(self, g):
        """(n_t, len(bc_dofs)) boundary values -- host array or CUDA tensor -- as a contiguous float64 device tensor."""
        shape = (self.n_t, int(self.bc_dofs.size))
        if isinstance(g, torch.Tensor) and g.is_cuda:
            g_dev = g.to(self.device, torch.float64).contiguous()
        else:
            g_dev = torch.from_numpy(np.ascontiguousarray(_as_host_f64(g), dtype=np.float64)).to(self.device)
        if g_dev.numel() != shape[0] * shape[1] or (g_dev.dim() == 2 and tuple(g_dev.shape) != shape):
            raise ValueError(f"bc values must have shape {shape} (n_t, len(bc_dofs))")
        return g_dev

    def lift_bc_device(self, g, b_dev, layout=L.CTL_LAYOUT_BLOCK_MAJOR):
        """Lift inhomogeneous Dirichlet data into the device right-hand side ``b_dev`` in place (``ctl_lift_bc``): the
        terms the reference adds through ``v_inhom`` (control/control.py:2993-3124 BE, 3137-3212 CN), with the K
        values the system holds, T_1 / T_2 applied, constrained rows untouched.  ``g``: (n_t, len(bc_dofs)) host array
        or CUDA tensor, columns in the order of ``bc_dofs`` (what ``Control.Instationary._dirichlet_data`` returns);
        every rank passes all of it.  Returns ``b_dev``."""
        self._check_vecs("lift_bc_device", b_dev, layout=layout)
        g_dev = self._bc_values_device(g)
        self._call(self._lib.ctl_lift_bc, g_dev.data_ptr(), b_dev.data_ptr(), layout)
        return b_dev

    def objective(self, v, zeta, v_hat):
        v = np.ascontiguousarray(v, dtype=np.float64)
        zeta = np.ascontiguousarray(zeta, dtype=np.float64)
        v_hat = np.ascontiguousarray(v_hat, dtype=np.float64)
        out = C.c_double()
        self._check(self._lib.ctl_objective_host(self._h, v.ctypes.data, zeta.ctypes.data,
                                                 v_hat.ctypes.data, C.byref(out)))
        return float(out.value)

    def micro_benchmarks(self, hierarchy=0, reps=10, flush_l2=True):
        """Isolated timings of the sweep kernels (CUDA events per launch)."""
        out = (C.c_double * 7)()
        self._call(self._lib.ctl_time_amg, hierarchy, reps, int(flush_l2), out)
        return {"cheb_ms": out[0], "cheb_bytes": out[1], "residual_ms": out[2], "residual_bytes": out[3],
                "inner_solve_ms": out[4], "inner_solve_bytes": out[5], "inner_solve_kernels": int(out[6]),
                "l2_flushed": bool(flush_l2)}

    def kernel_launches(self):
        return int(self._lib.ctl_kernel_launches(self._h))

    # ------------------------------------------------------------------ AMG introspection
    def amg_hierarchy(self, hierarchy=0):
        """Host copies of the level matrices: list of dicts with scipy CSR A, P and the
        aggregate ids (tests compare them with oracle/amg.py)."""
        import scipy.sparse as sp
        out = []
        nl = self._lib.ctl_amg_num_levels(self._h, hierarchy)
        for lvl in range(nl):
            n = C.c_int32()
            nnzA = C.c_int64()
            nnzP = C.c_int64()
            self._check(self._lib.ctl_amg_level_size(self._h, hierarchy, lvl, C.byref(n),
                                                     C.byref(nnzA), C.byref(nnzP)))
            entry = {"n": n.value}
            for which, nnz, key in ((0, nnzA.value, "A"), (1, nnzP.value, "P")):
                if nnz == 0:
                    entry[key] = None
                    continue
                ip = np.zeros(n.value + 1, dtype=np.int32)
                ix = np.zeros(nnz, dtype=np.int32)
                va = np.zeros(nnz, dtype=np.float64)
                self._check(self._lib.ctl_amg_get_csr(self._h, hierarchy, lvl, which,
                                                      ip.ctypes.data, ix.ctypes.data, va.ctypes.data))
                ncols = n.value if which == 0 else (int(ix.max()) + 1 if nnz else 0)
                entry[key] = (ip, ix, va, ncols)
            if entry["P"] is not None:
                agg = np.zeros(n.value, dtype=np.int32)
                self._check(self._lib.ctl_amg_get_aggregates(self._h, hierarchy, lvl, agg.ctypes.data))
                entry["agg"] = agg
            out.append(entry)
        for i, e in enumerate(out):
            ip, ix, va, _ = e["A"]
            e["A"] = sp.csr_matrix((va, ix, ip), shape=(e["n"], e["n"]))
            if e["P"] is not None:
                ip, ix, va, _ = e["P"]
                e["P"] = sp.csr_matrix((va, ix, ip), shape=(e["n"], out[i + 1]["n"]))
        return out

    def amg_solve(self, b_dev, hierarchy=0):
        x = torch.zeros_like(b_dev)
        self._call(self._lib.ctl_amg_solve, hierarchy, b_dev.data_ptr(), x.data_ptr())
        return x


class _DevPtr:
    """Raw device pointer exposed through __cuda_array_interface__ (zero-copy torch view)."""

    def __init__(self, ptr, count):
        self.__cuda_array_interface__ = {"shape": (count,), "typestr": "<f8",
                                         "data": (int(ptr), False), "version": 2}


def _wrap_device_ptr(ptr, count, device):
    return torch.as_tensor(_DevPtr(ptr, count), device=device)


class _MatShell:
    """petsc4py python-matrix context: ``mult(A, x, y)`` as at
    preconditioner/preconditioner.py:375-376.  ``x`` / ``y`` are PETSc Vecs (or anything
    with ``getArray`` / the numpy array interface) in the block-major layout; this
    compatibility path copies x to the device and y back on every call."""

    def __init__(self, system):
        self._s = system

    def mult(self, A, x, y):
        try:
            s = self._s
            xd = s.to_device(_as_host_f64(x))
            yd = s.apply(xd)
            np.copyto(_as_host_f64(y).reshape(-1), yd.cpu().numpy())
        except Exception:
            _error_flag[0] = True
            raise


class _PCShell:
    """petsc4py python-PC context: ``apply(pc, x, y)`` as at
    preconditioner/preconditioner.py:562-563."""

    def __init__(self, system, pc_fn=None):
        self._s = system
        self._pc_fn = pc_fn

    def apply(self, pc, x, y):
        try:
            s = self._s
            xh = np.asarray(_as_host_f64(x), dtype=np.float64).reshape(-1)
            if self._pc_fn is None:
                yd = s.pc_apply(s.to_device(xh))
                np.copyto(_as_host_f64(y).reshape(-1), yd.cpu().numpy())
                return
            # user callable: the nullspace wrapping of Preconditioner.apply on the host
            half = s.N * s.n_local
            b0 = xh[:half].reshape(s.N, s.n_local)
            b1 = xh[half:].reshape(s.N, s.n_local)
            b0c, b1c = b0.copy(), b1.copy()
            b0c[:, s.bc_dofs] = 0.0
            b1c[:, s.bc_dofs] = 0.0
            u0, u1 = np.zeros_like(b0), np.zeros_like(b1)
            self._pc_fn(u0, u1, b0c, b1c)
            u0[:, s.bc_dofs] = b0[:, s.bc_dofs]
            u1[:, s.bc_dofs] = b1[:, s.bc_dofs]
            np.copyto(_as_host_f64(y).reshape(-1), np.concatenate([u0.ravel(), u1.ravel()]))
        except Exception:
            _error_flag[0] = True
            raise
