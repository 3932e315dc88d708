"""Operator and preconditioner counts of the Krylov start (krylov.cuh, krylov_solve): from a zero guess the first
residual is b itself, so the solve skips the apply A 0 and, for MINRES and left-preconditioned GMRES, reuses the
preconditioned b of the reference norm.  A non-zero guess, and any guess under a user callback, keep PETSc's call
sequence.  fp64; tolerances are those of tests/test_gpu_pc.py."""
import numpy as np
import pytest

import kat
from oracle import control as ocontrol

pytestmark = pytest.mark.gpu

# at most one Krylov cycle (max_it < restart), so the counts below are exact; "preconditioner" returns an
# unconverged solve instead of raising
SP = {"gmres_restart": 30, "maximum_iterations": 29, "relative_tolerance": 1e-9, "absolute_tolerance": 0.0,
      "preconditioner": True, "monitor_convergence": False}
# extra operator / preconditioner applications over `its` when starting from a zero and from a non-zero guess
EXTRA = {"minres": ((0, 1), (1, 2)), "gmres": ((0, 1), (1, 2)), "fgmres": ((0, 0), (1, 0))}


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _setup(ksp):
    from control_b200 import MultiBlockSystem
    q = kat.heat_problem(16, 8, True)
    mode = "diagonal" if ksp == "minres" else "triangular"
    sp_ = dict(SP, linear_solver=ksp)
    ref = ocontrol.linear_solve(q["M"], q["K"], beta=q["beta"], n_t=q["n_t"], CN=True,
                                time_interval=q["time_interval"], bdofs=q["bdofs"], v_d=q["v_d"], f=q["f"],
                                lambda_v_bounds=q["lambda_v_bounds"], solver_parameters=sp_, pc_mode=mode)
    s = MultiBlockSystem(q["M"], q["K"], n_t=q["n_t"], beta=q["beta"], CN=True, time_interval=q["time_interval"],
                         bc_dofs=q["bdofs"])
    s.setup_preconditioner(lambda_v_bounds=q["lambda_v_bounds"], mode=mode)
    return s, sp_, ref


@pytest.mark.parametrize("ksp", ["minres", "gmres", "fgmres"])
def test_zero_guess_skips_the_repeated_start(ksp):
    s, sp_, ref = _setup(ksp)
    (zm, zp), (nm, np_) = EXTRA[ksp]
    u0, u1 = np.zeros((s.N, s.n)), np.zeros((s.N, s.n))
    info = s.solve(u0, u1, ref["b_0"], ref["b_1"], solver_parameters=sp_, pc_fn="builtin")
    assert info.reason == ref["ksp"].reason and abs(info.its - ref["ksp"].its) <= 1
    assert (info.n_mult, info.n_pc) == (info.its + zm, info.its + zp)
    k = min(len(info.history), len(ref["ksp"].history)) - 1
    assert np.allclose(info.history[:k], ref["ksp"].history[:k], rtol=1e-6)
    assert _rel(u0, ref["v_blocks"]) < 1e-7 and _rel(u1, ref["zeta_blocks"]) < 1e-7
    # non-zero guesses take the full start; 1e-170 squares to zero, so a sum of squares would call it zero
    rng = np.random.default_rng(1)
    for scale in (1e-3, 1e-170):
        g0, g1 = scale * rng.standard_normal((s.N, s.n)), scale * rng.standard_normal((s.N, s.n))
        info = s.solve(g0, g1, ref["b_0"], ref["b_1"], solver_parameters=sp_, pc_fn="builtin")
        assert (info.n_mult, info.n_pc) == (info.its + nm, info.its + np_), scale
    s.close()


@pytest.mark.parametrize("ksp", ["minres", "gmres"])
def test_user_callback_keeps_the_full_start(ksp):
    s, sp_, ref = _setup(ksp)
    inner = s.pc_fn()
    calls = []

    def P(u_0, u_1, b_0, b_1):
        calls.append(1)
        inner(u_0, u_1, b_0, b_1)

    u0, u1 = np.zeros((s.N, s.n)), np.zeros((s.N, s.n))
    info = s.solve(u0, u1, ref["b_0"], ref["b_1"], solver_parameters=sp_, pc_fn=P)
    assert info.reason > 0 and abs(info.its - ref["ksp"].its) <= 1
    assert (info.n_mult, info.n_pc) == (info.its + 1, info.its + 2) and len(calls) == info.n_pc
    assert _rel(u0, ref["v_blocks"]) < 1e-7 and _rel(u1, ref["zeta_blocks"]) < 1e-7
    s.close()
