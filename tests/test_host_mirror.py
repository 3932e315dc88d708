"""Host logic of the ``Control`` mirror WITHOUT a GPU: the device systems (``MultiBlockSystem``, ``StokesSystem``)
are replaced, for the duration of a test, by stand-ins that solve the same block systems with the oracle, so
that everything the host side does around a solve -- right-hand sides, lifting of boundary data, the
stationary-to-trapezoidal mapping, unpacking, residuals and updates of the Picard / Gauss-Newton loops, the
pressure-space forward matrices of the Navier-Stokes loop -- is compared with the oracle's own restatement of
the reference drivers.  (The product never does this: without a GPU ``MultiBlockSystem`` raises; the same
drivers run against the real device systems in the ``-m gpu`` tests.)"""
import numpy as np
import pytest

import kat
from oracle import control as ocontrol
from oracle import kkt, stationary, stokes
from oracle.pc import construct_pc
from synthetic import fem


class _Info:
    def __init__(self, res):
        self.its, self.reason, self.history = res.its, res.reason, list(res.history)


class FakeMultiBlockSystem:
    """The calls ``control_b200.control`` / ``control_b200.stationary`` make on a ``MultiBlockSystem``."""

    def __init__(self, M, K, *, n_t, beta, CN, time_interval=(0.0, 1.0), bc_dofs=(), device=None, rank=0, world=1):
        self.M, self.K, self.n_t, self.beta, self.CN = M, K, n_t, beta, CN
        self.tau = (time_interval[1] - time_interval[0]) / (n_t - 1.0)
        self.bd = np.asarray(bc_dofs, dtype=np.int64)
        self.n = self.n_local = M.shape[0]
        self.N = kkt.n_blocks(n_t, CN)
        self.row_begin, self.world = 0, 1
        self.pc = None

    def set_K(self, K):
        self.K, self.pc = K, None

    def setup_preconditioner(self, *, lambda_v_bounds=None, Multigrid=False, mode="triangular", **amg):
        assert mode == "triangular"
        self.pc = construct_pc(self.M, self.K, self.tau, self.beta, self.n_t, self.CN, self.bd,
                               lambda_v_bounds=lambda_v_bounds, Multigrid=Multigrid, amg_params=amg or None)

    def solve(self, u_0, u_1, b_0, b_1, *, solver_parameters, pc_fn):
        assert pc_fn == "builtin" and self.pc is not None
        v, z, res = ocontrol.system_solve(
            lambda x0, x1: kkt.kkt_apply_fused(self.M, self.K, self.tau, self.beta, self.n_t, self.CN, self.bd, x0, x1),
            kkt.DirichletBCNullspace(self.bd), u_0, u_1, b_0, b_1, solver_parameters=solver_parameters, pc_fn=self.pc)
        u_0[:], u_1[:] = v, z
        return _Info(res)

    def close(self):
        pass


class FakeStokesSystem:
    """The calls ``Control.Instationary.incompressible_*`` make on a ``StokesSystem``."""

    def __init__(self, M_v, K_v, B, M_p, K_p, *, n_t, beta, CN, time_interval=(0.0, 1.0), bc_dofs_v=(), device=None,
                 D_p=None):
        self.a = dict(M_v=M_v, K_v=K_v, B=B, M_p=M_p, K_p=K_p)
        self.kw = dict(beta=beta, n_t=n_t, CN=CN, time_interval=time_interval, bdofs_v=np.asarray(bc_dofs_v, dtype=np.int64))
        self.D_p = D_p
        self.pc_kw = None

    def set_forward(self, K_v, D_p=None):
        self.a["K_v"] = K_v
        if D_p is not None:
            assert self.D_p is not None
            self.D_p = D_p
        self.pc_kw = None

    def setup_preconditioner(self, *, lambda_v_bounds=None, lambda_p_bounds=None, amg=None, amg_p=None, Multigrid=False):
        self.pc_kw = dict(lambda_v_bounds=lambda_v_bounds, lambda_p_bounds=lambda_p_bounds, amg_params=amg, amg_params_p=amg_p,
                          Multigrid=Multigrid)

    def solve(self, u_0, u_1, b_0, b_1, *, solver_parameters, pc_fn):
        assert pc_fn == "builtin" and self.pc_kw is not None
        w0, w1, res = stokes.stokes_solve(self.a["M_v"], self.a["K_v"], self.a["B"], self.a["M_p"], self.a["K_p"],
                                          b_0=b_0, b_1=b_1, solver_parameters=solver_parameters, D_p=self.D_p,
                                          **self.kw, **self.pc_kw)
        u_0[:], u_1[:] = w0, w1
        return _Info(res)

    def close(self):
        pass


@pytest.fixture
def fake_device(monkeypatch):
    import control_b200.control as cc
    import control_b200.stationary as cs
    import control_b200.stokes as cst
    monkeypatch.setattr(cc, "MultiBlockSystem", FakeMultiBlockSystem)
    monkeypatch.setattr(cs, "MultiBlockSystem", FakeMultiBlockSystem)
    monkeypatch.setattr(cst, "StokesSystem", FakeStokesSystem)
    from control_b200 import Control
    return Control


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


SP = {"linear_solver": "fgmres", "maximum_iterations": 200, "relative_tolerance": 1e-10, "absolute_tolerance": 0.0}


def test_stationary_driver_host_logic(fake_device):
    """``Control.Stationary`` (mapping onto n_t = 2, tau = 2, K' = D_v - M; lifting; Picard and Gauss-Newton
    loops) against the direct restatement of control/control.py:351-800 in oracle/stationary.py."""
    Control = fake_device
    nx = 8
    M, L, coords, bd = fem.assemble_p1_2d(nx, nx, 1.0, 1.0)
    x, y = coords[:, 0], coords[:, 1]
    v_hat = np.sin(np.pi * x) * np.sin(np.pi * y) * np.exp(x + y)
    beta = 1e-2
    D_v = (L + 2.0 * M).tocsr()
    g = np.cos(3.0 * x[bd]) + y[bd]
    f = M @ (x * y)
    c = Control.Stationary(M, D_v, desired_state=lambda: (M @ v_hat, v_hat), force_f=lambda: f, beta=beta, bc_dofs=bd,
                           bc_values=g)
    info = c.linear_solve(solver_parameters=SP, lambda_v_bounds=(0.5, 2.0), print_error=False)
    ref = stationary.linear_solve(M, D_v, beta=beta, bdofs=bd, v_d=M @ v_hat, f=f, bc_values=g, solver_parameters=SP,
                                  lambda_v_bounds=(0.5, 2.0))
    assert info.its == ref["ksp"].its
    assert _rel(c._v, ref["v"]) < 1e-9 and _rel(c._zeta, ref["zeta"]) < 1e-9
    D = fem.nonlinear_diffusion_p1_2d(nx, nx, 1.0, 1.0)
    for gauss_newton in (False, True):
        c = Control.Stationary(M, D, desired_state=lambda: (M @ v_hat, v_hat), beta=beta, Gauss_Newton=gauss_newton,
                               bc_dofs=bd)
        k = c.non_linear_solve(solver_parameters=SP, lambda_v_bounds=(0.5, 2.0), max_non_linear_iter=30,
                               print_error_non_linear=False)
        out = stationary.non_linear_solve(M, lambda v: D(v, gauss_newton), beta=beta, bdofs=bd, v_d=M @ v_hat,
                                          f=np.zeros(M.shape[0]), solver_parameters=SP, lambda_v_bounds=(0.5, 2.0),
                                          max_non_linear_iter=30)
        assert k == out["iterations"]
        assert np.allclose(c.non_linear_history, out["history"], rtol=1e-6)
        assert _rel(c._v, out["v"]) < 1e-8


@pytest.mark.parametrize("CN", [True, False])
def test_instationary_convection_diffusion_host_logic(fake_device, CN):
    """``Control.Instationary.linear_solve`` with a time-dependent non-symmetric forward matrix and
    inhomogeneous Dirichlet data (the reference's convection-diffusion studies) against oracle/control.py."""
    Control = fake_device
    q = kat.mms_convection_diffusion_problem(4, 12, CN)

    def level(t):
        return int(round(t / q["tau"]))
    c = Control.Instationary(q["M"], lambda v_i, t, gauss_newton: q["K_levels"][level(t)],
                             desired_state=lambda t: (q["v_d"][level(t)], q["v_hat"][level(t)]),
                             force_f=lambda t: q["f"][level(t)], beta=q["beta"], n_t=q["n_t"], CN=CN,
                             time_interval=q["time_interval"], bc_dofs=q["bdofs"],
                             bc_values=lambda t: q["bc_values"][level(t)], initial_condition=q["v_0"])
    info = c.linear_solve(solver_parameters=SP, lambda_v_bounds=(0.5, 2.0), print_error=False)
    ref = ocontrol.linear_solve(q["M"], q["K_levels"], beta=q["beta"], n_t=q["n_t"], CN=CN,
                                time_interval=q["time_interval"], bdofs=q["bdofs"], v_d=q["v_d"], f=q["f"], v_0=q["v_0"],
                                bc_values=q["bc_values"], solver_parameters=SP, lambda_v_bounds=(0.5, 2.0))
    assert info.its == ref["ksp"].its
    assert _rel(c._v, ref["v"]) < 1e-9 and _rel(c._zeta, ref["zeta"]) < 1e-9


@pytest.mark.parametrize("CN", [True, False])
def test_navier_stokes_picard_loop_host_logic(fake_device, CN):
    """``Control.Instationary.incompressible_non_linear_solve`` (control/control.py:4886-5219) on the problem of
    the reference's Navier-Stokes tests (4 x 4 cells): residual history, inner iteration counts and iterates
    against oracle/stokes.py::incompressible_non_linear_solve."""
    Control = fake_device
    q = kat.reference_navier_stokes_problem(CN, nx=4, n_t=6)
    sq = q["sq"]

    def level(t):
        return int(round(t / q["tau"]))
    c = Control.Instationary(q["M"], lambda v_i, t, gauss_newton: q["D_v"](v_i, t),
                             desired_state=lambda t: (q["v_d"][level(t)], q["v_hat"][level(t)]), beta=q["beta"],
                             n_t=q["n_t"], CN=CN, time_interval=q["time_interval"], bc_dofs=q["bdofs"],
                             bc_values=lambda t: q["bc_values"][level(t)])
    space_p = dict(B=q["B"], M_p=sq["M_p"], K_p=sq["L_p"], forward_matrix_p=lambda v_i, t, gauss_newton: q["D_p"](v_i, t))
    sp_ = dict(SP, relative_tolerance=1e-8)
    k = c.incompressible_non_linear_solve("constant", space_p=space_p, solver_parameters=sp_,
                                          lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"],
                                          print_error_non_linear=False)
    out = stokes.incompressible_non_linear_solve(
        q["M"], q["D_v"], q["B"], sq["M_p"], sq["L_p"], q["D_p"], beta=q["beta"], n_t=q["n_t"], CN=CN,
        time_interval=q["time_interval"], bdofs_v=q["bdofs"], v_d=q["v_d"], f=q["f"], bc_values=q["bc_values"],
        solver_parameters=sp_, lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"])
    assert k == out["iterations"] and k >= 3
    assert c.inner_iterations == out["inner_its"]
    assert np.allclose(c.non_linear_history, out["history"], rtol=1e-8)
    assert out["history"][-1] <= 1e-5 * out["history"][0]
    assert _rel(c._v, out["v"]) < 1e-9 and _rel(c._zeta, out["zeta"]) < 1e-9
    assert _rel(c._p, out["p"]) < 1e-8 and _rel(c._mu, out["mu"]) < 1e-8
    assert np.array_equal(c._v[:, q["bdofs"]], q["bc_values"])


def _stationary_stokes_kat():
    """test/test_control.py:232-358: vector Q2 - Q1 on 4 x 4 quads, forward form grad.grad + mass, analytic fields."""
    sq = fem.assemble_q2q1_stokes_2d(4, 4)
    M, L, B, Mp, Lp = sq["M_v"], sq["L_v"], sq["B"], sq["M_p"], sq["L_p"]
    K = (L + M).tocsr()
    beta = 1e-3
    x, y = sq["coords_v"][:, 0], sq["coords_v"][:, 1]
    px, py = sq["coords_p"][:, 0], sq["coords_p"][:, 1]

    def vec(cx, cy):
        a = np.zeros(M.shape[0])
        a[0::2], a[1::2] = cx, cy
        return a
    v_ref = vec(x * np.exp(y) * np.sin(np.pi * x) * np.sin(2.0 * np.pi * y), np.sin(3.0 * np.pi * x) * np.sin(4.0 * np.pi * y))
    zeta_ref = vec(np.sin(np.pi * x) * np.sin(2.0 * np.pi * y), np.sin(3.0 * np.pi * x) * np.sin(4.0 * np.pi * y))
    p_ref = np.sin(np.pi * px) * np.sin(2.0 * np.pi * py)
    mu_ref = px * np.exp(py)
    rhs = dict(v_d=M @ v_ref + K @ zeta_ref + B.T @ mu_ref, f=K @ v_ref - (1.0 / beta) * (M @ zeta_ref) + B.T @ p_ref,
               div_v=B @ v_ref, div_zeta=B @ zeta_ref)
    return dict(sq=sq, M=M, K=K, B=B, Mp=Mp, Lp=Lp, D_p=(Lp + Mp).tocsr(), beta=beta, rhs=rhs, v_ref=v_ref,
                zeta_ref=zeta_ref, p_ref=p_ref, mu_ref=mu_ref, bd=sq["bdofs_v"])


def test_stationary_stokes_known_answer_through_both_drivers(fake_device):
    """The reference's stationary Stokes known-answer test through (a) the oracle's literal restatement of
    ``Stationary.incompressible_linear_solve`` and (b) the host mirror, which maps the system onto the
    instationary Stokes handle (one block, tau = 2, shifted forward matrices, divergence rows scaled by 2):
    both reproduce the analytic fields (the reference asserts 1e-13; 5e-13 here, the attainable error at
    rtol 1e-14), and agree with each other."""
    Control = fake_device
    k = _stationary_stokes_kat()
    sp_ = {"linear_solver": "fgmres", "fgmres_restart": 10, "maximum_iterations": 500, "relative_tolerance": 1e-14,
           "absolute_tolerance": 1e-14}
    bounds = dict(lambda_v_bounds=(0.3924, 2.0598), lambda_p_bounds=(0.5, 2.0))
    v, zeta, p, mu, res = stationary.incompressible_linear_solve(
        k["M"], k["K"], k["B"], k["Mp"], k["Lp"], beta=k["beta"], bdofs_v=k["bd"], D_p=k["D_p"], check_v_d=False,
        check_f=False, solver_parameters=sp_, **bounds, **k["rhs"])
    c = Control.Stationary(k["M"], k["K"], beta=k["beta"], bc_dofs=k["bd"])
    space_p = dict(B=k["B"], M_p=k["Mp"], K_p=k["Lp"], forward_matrix_p=k["D_p"])
    info = c.incompressible_linear_solve("constant", space_p=space_p, solver_parameters=sp_, print_error=False,
                                         **bounds, **k["rhs"])
    assert res.reason > 0 and info.reason > 0 and abs(info.its - res.its) <= 3
    M, Mp = k["M"], k["Mp"]

    def shift(q):                                             # test/test_control.py:334-347
        return q - np.ones(Mp.shape[0]) @ (Mp @ q)
    for vv, zz, pp, mm in ((v, zeta, p, mu), (c._v, c._zeta, c._p, c._mu)):
        assert kat.l2_error(M, vv[None], k["v_ref"][None]) < 5e-13
        assert kat.l2_error(M, zz[None], k["zeta_ref"][None]) < 5e-13
        # pressures: the Krylov solve stops at 1e-14 x |b| with |b| ~ 1/beta = 1e3 (measured errors up to 9e-13; the
        # dense direct solve of the same operator in tests/test_oracle.py reaches the reference's 1e-13)
        assert kat.l2_error(Mp, shift(pp)[None], shift(k["p_ref"])[None]) < 3e-12
        assert kat.l2_error(Mp, shift(mm)[None], shift(k["mu_ref"])[None]) < 3e-12


def test_stationary_navier_stokes_picard_loop_host_logic(fake_device):
    """``Stationary.incompressible_non_linear_solve`` (control/control.py:1203-1486), lid-driven cavity with the
    forward form of the reference's Navier-Stokes tests, host mirror (mapped onto the instationary handle)
    against the oracle's literal restatement."""
    Control = fake_device
    q = kat.reference_navier_stokes_problem(True, nx=4)
    sq = q["sq"]
    g = q["bc_values"][-1]
    v_d, v_hat = q["v_d"][0], q["v_hat"][0]
    sp_ = dict(SP, relative_tolerance=1e-9)
    bounds = dict(lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"])
    out = stationary.incompressible_non_linear_solve(
        q["M"], lambda v: q["D_v"](v, 0.0), q["B"], sq["M_p"], sq["L_p"], lambda v: q["D_p"](v, 0.0), beta=q["beta"],
        bdofs_v=q["bdofs"], v_d=v_d, f=np.zeros(q["M"].shape[0]), bc_values=g, solver_parameters=sp_, **bounds)
    c = Control.Stationary(q["M"], lambda v, gauss_newton: q["D_v"](v, 0.0), desired_state=lambda: (v_d, v_hat),
                           beta=q["beta"], bc_dofs=q["bdofs"], bc_values=g)
    space_p = dict(B=q["B"], M_p=sq["M_p"], K_p=sq["L_p"], forward_matrix_p=lambda v, gauss_newton: q["D_p"](v, 0.0))
    k = c.incompressible_non_linear_solve("constant", space_p=space_p, solver_parameters=sp_,
                                          print_error_non_linear=False, **bounds)
    assert k == out["iterations"] and out["history"][-1] <= 1e-5 * out["history"][0]
    assert np.allclose(c.non_linear_history, out["history"], rtol=1e-4)
    assert _rel(c._v, out["v"]) < 1e-6 and _rel(c._zeta, out["zeta"]) < 1e-6
    pm = out["p"] - out["p"].mean()
    assert np.abs((c._p - c._p.mean()) - pm).max() < 1e-5 * np.abs(pm).max()


@pytest.mark.parametrize("CN,gauss_newton", [(True, False), (False, False), (True, True)])
def test_instationary_non_linear_loop_with_inhomogeneous_data_host_logic(fake_device, CN, gauss_newton):
    """``Control.Instationary.non_linear_solve`` (control/control.py:3377-3590) with time-dependent inhomogeneous
    Dirichlet data (re-imposed on the iterate after every update, 3480-3483) and the non-linear diffusion
    operator of BASELINE config C5, against oracle/control.py::non_linear_solve."""
    Control = fake_device
    nx, n_t = 6, 5
    q = kat.heat_problem(nx, n_t, CN, beta=1e-2)
    Dv = fem.nonlinear_diffusion_p1_2d(nx, nx, 2.0, 2.0)
    times = q["tau"] * np.arange(n_t)
    xb, yb = q["coords"][q["bdofs"], 0], q["coords"][q["bdofs"], 1]
    g = 0.3 * np.stack([np.cos(xb + t) + 0.5 * yb for t in times])

    def level(t):
        return int(round(t / q["tau"]))
    c = Control.Instationary(q["M"], lambda v, t, gn: Dv(v, gn), desired_state=lambda t: (q["v_d"][level(t)], q["v_hat"][level(t)]),
                             force_f=lambda t: q["f"][level(t)], beta=q["beta"], Gauss_Newton=gauss_newton, n_t=n_t,
                             CN=CN, time_interval=q["time_interval"], bc_dofs=q["bdofs"],
                             bc_values=lambda t: g[level(t)])
    k = c.non_linear_solve(lambda_v_bounds=q["lambda_v_bounds"], solver_parameters=SP, max_non_linear_iter=6,
                           print_error_non_linear=False)
    ref = ocontrol.non_linear_solve(q["M"], lambda v, t: Dv(v, gauss_newton), beta=q["beta"], n_t=n_t, CN=CN,
                                    time_interval=q["time_interval"], bdofs=q["bdofs"], v_d=q["v_d"], f=q["f"],
                                    solver_parameters=SP, lambda_v_bounds=q["lambda_v_bounds"], max_non_linear_iter=6,
                                    bc_values=g)
    assert k == ref["iterations"] and k >= 2
    assert np.allclose(c.non_linear_history, ref["history"], rtol=1e-8)
    assert _rel(c._v, ref["v"]) < 1e-9 and _rel(c._zeta, ref["zeta"]) < 1e-9
    assert np.array_equal(c._v[1:, q["bdofs"]], g[1:])
    if not gauss_newton:                                  # (the Gauss-Newton variant of the reference evaluates the
        assert ref["history"][-1] < 0.2 * ref["history"][0]   # residual with the Jacobian, DESIGN.md section 1 row a11)


def _loop_lines(history):
    return [f"Initial non-linear residual: {history[0]:.16e}"] + \
        [f"Non-linear solver: iteration {k:d}, non-linear residual norm {h:.16e}" for k, h in enumerate(history[1:], 1)]


def test_outer_loop_output(fake_device, capsys):
    """What a heat and a Navier-Stokes loop print with ``print_error_non_linear``: the first residual norm, then one
    line per outer iteration, formatted as the reference's loops (control/control.py:3377-3590, 4886-5219) format
    them, and nothing else when the inner solves are quiet; ``max_non_linear_iter`` stops both after the second."""
    Control = fake_device
    quiet = dict(SP, monitor_convergence=False)
    q = kat.heat_problem(6, 5, True, beta=1e-2)
    Dv = fem.nonlinear_diffusion_p1_2d(6, 6, 2.0, 2.0)

    def level(t):
        return int(round(t / q["tau"]))
    c = Control.Instationary(q["M"], lambda v, t, gn: Dv(v, gn), desired_state=lambda t: (q["v_d"][level(t)], q["v_hat"][level(t)]),
                             force_f=lambda t: q["f"][level(t)], beta=q["beta"], n_t=5, CN=True,
                             time_interval=q["time_interval"], bc_dofs=q["bdofs"])
    capsys.readouterr()
    k = c.non_linear_solve(lambda_v_bounds=q["lambda_v_bounds"], solver_parameters=quiet, max_non_linear_iter=2,
                           print_error_non_linear=True, device_loop=False)
    assert k == 2 and len(c.non_linear_history) == 3
    assert capsys.readouterr().out.splitlines() == _loop_lines(c.non_linear_history)

    q = kat.reference_navier_stokes_problem(False, nx=4, n_t=6)
    sq = q["sq"]

    def level(t):
        return int(round(t / q["tau"]))
    c = Control.Instationary(q["M"], lambda v_i, t, gn: q["D_v"](v_i, t),
                             desired_state=lambda t: (q["v_d"][level(t)], q["v_hat"][level(t)]), beta=q["beta"],
                             n_t=q["n_t"], CN=False, time_interval=q["time_interval"], bc_dofs=q["bdofs"],
                             bc_values=lambda t: q["bc_values"][level(t)])
    space_p = dict(B=q["B"], M_p=sq["M_p"], K_p=sq["L_p"], forward_matrix_p=lambda v_i, t, gn: q["D_p"](v_i, t))
    capsys.readouterr()
    k = c.incompressible_non_linear_solve("constant", space_p=space_p, solver_parameters=quiet, max_non_linear_iter=2,
                                          lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"])
    assert k == 2 and len(c.non_linear_history) == 3 and len(c.inner_iterations) == 2
    assert capsys.readouterr().out.splitlines() == _loop_lines(c.non_linear_history)
