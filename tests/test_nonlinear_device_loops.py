"""Device-resident non-linear loops: the Navier-Stokes Picard loop on ctl_stokes_nonlinear_residual, and the heat-type
Picard / Gauss-Newton loop with inhomogeneous Dirichlet data, both behind ``device_loop=True`` of the drivers.

CPU: the reference's Navier-Stokes residual (res_eval) equals the lifted right-hand side minus the outer operator with
RAW coupling products -- and not minus the nullspace-corrected operator of ctl_stokes_apply -- and its norm is the
T^-1 / tau formula; ``device_loop=True`` refuses ``P=`` and several ranks before any device work.  GPU: the residual
kernel against the host residual, both drivers against the oracle and the NS driver against its own host loop, and the
argument / state errors of the new entry point."""
import ctypes as C

import numpy as np
import pytest

import kat
from oracle import control as ocontrol
from oracle import kkt
from oracle import stokes as ostokes
from synthetic import fem

SEED = 20261021


def _T_v(y, N, CN):
    """T of the velocity rows: T_1 on the first N blocks, T_2 on the next N."""
    return np.concatenate([kkt.apply_T_1(y[:N]), kkt.apply_T_2(y[N:])]) if CN else y.copy()


def _T_p(y, N, CN):
    """T of the pressure rows: T_2 on the first N blocks (the rows of B v), T_1 on the next N (B zeta)."""
    return np.concatenate([kkt.apply_T_2(y[:N]), kkt.apply_T_1(y[N:])]) if CN else y.copy()


def _reference_norm_of(r0, r1, N, tau, CN):
    """sqrt(||T^-1 r_v||^2 + ||T^-1 r_p||^2 / tau^2) of a transformed outer residual."""
    if CN:
        r0 = np.concatenate([kkt.apply_T_1_inv(r0[:N]), kkt.apply_T_2_inv(r0[N:])])
        r1 = np.concatenate([kkt.apply_T_2_inv(r1[:N]), kkt.apply_T_1_inv(r1[N:])])
    return float(np.sqrt((r0 ** 2).sum() + (r1 ** 2).sum() / tau ** 2))


def _ns_case(CN, nx=4, n_t=6, seed=SEED):
    """The lid-driven cavity of the reference's Navier-Stokes tests at a Picard iterate as the loop leaves it: g on the
    constrained velocity dofs of every level (for CN level 0 is the initial condition, so it carries g_0 too), random
    zeta with zero boundary rows, and mu, p with clearly nonzero per-block means.  Returns the problem, the iterate,
    the reference's residual parts (res_eval, oracle/stokes.py) in transformed form, their norm, the homogeneous
    velocity rows of b and the per-level D_v_i / D_p_i."""
    from control_b200.control import build_rhs
    rng = np.random.default_rng(seed)
    q = kat.reference_navier_stokes_problem(CN, nx=nx, n_t=n_t)
    M, B, bd, tau, beta = q["M"], q["B"], q["bdofs"], q["tau"], q["beta"]
    N = n_t - 1 if CN else n_t
    n_v, n_p = M.shape[0], q["sq"]["M_p"].shape[0]
    times = tau * np.arange(n_t)
    g = q["bc_values"]
    v_old = 0.2 * rng.standard_normal((n_t, n_v))
    v_old[:, bd] = g
    zeta_old = rng.standard_normal((n_t, n_v))
    zeta_old[:, bd] = 0.0
    v_0 = np.zeros(n_v)
    if CN:
        zeta_old[-1] = 0.0
        v_0 = v_old[0].copy()
    mu = rng.standard_normal((N, n_p)) + 0.7 + np.arange(N)[:, None]
    p = rng.standard_normal((N, n_p)) - 1.3 + 0.5 * np.arange(N)[:, None]
    # res_eval of incompressible_non_linear_solve (control/control.py:4979-5072)
    r00, r01 = ocontrol.non_linear_res_eval(M, q["D_v"], times, tau, beta, n_t, CN, bd, v_old, zeta_old, v_0, q["v_d"],
                                            q["f"])
    r00 -= tau * (B.T @ mu.T).T
    r01 -= tau * (B.T @ p.T).T
    r00[:, bd] = 0.0
    r01[:, bd] = 0.0
    r10 = -(B @ (v_old[1:] if CN else v_old).T).T
    r11 = -(B @ (zeta_old[:-1] if CN else zeta_old).T).T
    ref_norm = float(np.sqrt(sum((a ** 2).sum() for a in (r00, r01, r10, r11))))
    # what incompressible_linear_solve makes of them: T on the velocity rows, div_v = tau r10, div_zeta = tau r11
    e0 = _T_v(np.concatenate([r00, r01]), N, CN)
    e1 = _T_p(tau * np.concatenate([r10, r11]), N, CN)
    K_it = [q["D_v"](v_old[i], times[i]) for i in range(n_t)]
    P_it = [q["D_p"](v_old[i], times[i]) for i in range(n_t)]
    b00, b01 = build_rhs(M, q["D_v"](v_0, times[0]), tau, n_t, CN, bd, q["v_d"], q["f"], v_0)
    x0 = np.concatenate([v_old[1:], zeta_old[:-1]] if CN else [v_old, zeta_old])
    x1 = np.concatenate([mu, p])
    return dict(q=q, N=N, n_v=n_v, n_p=n_p, g=g, v_0=v_0, x0=x0, x1=x1, e0=e0, e1=e1, ref_norm=ref_norm,
                b_hom=(np.concatenate([b00, b01]), np.zeros((2 * N, n_p))), K_it=K_it, P_it=P_it)


def _host_lifted_b(c):
    """The homogeneous b lifted with g on the host: velocity rows as build_rhs(bc_values=g) with the K_i of the
    iterate, divergence rows b_1_0 = -tau T_2(B g) (control/control.py:4107-4119, 4207-4219)."""
    from control_b200.control import build_rhs
    q, N, g = c["q"], c["N"], c["g"]
    M, B, bd, tau, n_t, CN = q["M"], q["B"], q["bdofs"], q["tau"], q["n_t"], q["CN"]
    z = np.zeros((n_t, M.shape[0]))
    args = (M, c["K_it"][0], tau, n_t, CN, bd, z, z, np.zeros(M.shape[0]))
    a, h = build_rhs(*args, bc_values=g, K_levels=c["K_it"]), build_rhs(*args, K_levels=c["K_it"])
    b0 = c["b_hom"][0] + np.concatenate([a[0] - h[0], a[1] - h[1]])
    lift = np.zeros((n_t, M.shape[0]))
    lift[:, bd] = g
    b1 = np.zeros_like(c["b_hom"][1])
    b1[:N] = -tau * (B @ (lift[1:] if CN else lift).T).T
    return b0, _T_p(b1, N, CN)


def _raw_operator(c):
    """A_raw x from oracle pieces: the fused heat KKT apply on the velocity blocks plus tau T(B^T x_p) on the velocity
    rows and tau T(B x_v) on the pressure rows, with no nullspace corrections."""
    q, N = c["q"], c["N"]
    M, B, bd, tau, n_t, CN = q["M"], q["B"], q["bdofs"], q["tau"], q["n_t"], q["CN"]
    x0, x1 = c["x0"], c["x1"]
    y0a, y0b = kkt.kkt_apply_fused(M, c["K_it"], tau, q["beta"], n_t, CN, bd, x0[:N], x0[N:])
    xc0 = x0.copy()
    xc0[:, bd] = 0.0
    g0 = _T_v(tau * (B.T @ x1.T).T, N, CN)
    g0[:, bd] = 0.0
    return np.concatenate([y0a, y0b]) + g0, _T_p(tau * (B @ xc0.T).T, N, CN)


# ---------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("CN", [True, False])
def test_navier_stokes_residual_is_lifted_rhs_minus_raw_operator(CN):
    c = _ns_case(CN)
    bd, N, tau = c["q"]["bdofs"], c["N"], c["q"]["tau"]
    b0, b1 = _host_lifted_b(c)
    y0, y1 = _raw_operator(c)
    d0, d1 = b0 - y0, b1 - y1
    d0[:, bd] = 0.0
    scale = max(np.abs(c["e0"]).max(), np.abs(c["e1"]).max())
    assert np.abs(d0 - c["e0"]).max() <= 1e-12 * scale
    assert np.abs(d1 - c["e1"]).max() <= 1e-12 * scale
    assert abs(_reference_norm_of(d0, d1, N, tau, CN) - c["ref_norm"]) <= 1e-12 * c["ref_norm"]
    # the operator of ctl_stokes_apply centres the pressure parts: with mu and p carrying per-block means its residual
    # is a different vector, which is why the loop needs a residual of its own
    q = c["q"]
    z0, z1 = ostokes.stokes_apply_fused(q["M"], c["K_it"], q["B"], tau, q["beta"], q["n_t"], CN, bd, c["x0"], c["x1"])
    w0, w1 = b0 - z0, b1 - z1
    w0[:, bd] = 0.0
    assert max(np.abs(w0 - c["e0"]).max(), np.abs(w1 - c["e1"]).max()) > 1e-6 * scale


def _heat_control(q, Dv, g, CN, gauss_newton, **kw):
    from control_b200 import Control

    def level(t):
        return int(round(t / q["tau"]))
    return Control.Instationary(q["M"], lambda v, t, gn: Dv(v, gn), desired_state=lambda t: (q["v_d"][level(t)],) * 2,
                                force_f=lambda t: q["f"][level(t)], beta=q["beta"], Gauss_Newton=gauss_newton, CN=CN,
                                n_t=q["n_t"], time_interval=q["time_interval"], bc_dofs=q["bdofs"],
                                bc_values=None if g is None else (lambda t: g[level(t)]), **kw)


def _ns_control(q):
    from control_b200 import Control

    def level(t):
        return int(round(t / q["tau"]))
    c = Control.Instationary(q["M"], lambda v_i, t, gauss_newton: q["D_v"](v_i, t),
                             desired_state=lambda t: (q["v_d"][level(t)], q["v_hat"][level(t)]), beta=q["beta"],
                             n_t=q["n_t"], CN=q["CN"], time_interval=q["time_interval"], bc_dofs=q["bdofs"],
                             bc_values=lambda t: q["bc_values"][level(t)])
    space_p = dict(B=q["B"], M_p=q["sq"]["M_p"], K_p=q["sq"]["L_p"],
                   forward_matrix_p=lambda v_i, t, gauss_newton: q["D_p"](v_i, t))
    return c, space_p


def test_device_loop_argument_errors_precede_device_work():
    q = kat.heat_problem(4, 4, True, beta=1e-2)
    Dv = fem.nonlinear_diffusion_p1_2d(4, 4, 2.0, 2.0)

    def P(u_0, u_1, b_0, b_1):
        raise AssertionError("never called")
    c = _heat_control(q, Dv, None, True, False)
    with pytest.raises(ValueError, match="P="):
        c.non_linear_solve(P=P, device_loop=True, print_error_non_linear=False)
    assert c._system is None
    c2 = _heat_control(q, Dv, None, True, False, world=2)
    with pytest.raises(ValueError, match="one rank"):
        c2.non_linear_solve(device_loop=True, print_error_non_linear=False)
    assert c2._system is None
    ns, space_p = _ns_control(kat.reference_navier_stokes_problem(True, nx=2, n_t=3))
    with pytest.raises(ValueError, match="P="):
        ns.incompressible_non_linear_solve("constant", space_p=space_p, P=P, device_loop=True,
                                           print_error_non_linear=False)
    assert getattr(ns, "_stokes", None) is None and ns._system is None


# ---------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("CN,n_t", [(True, 6), (False, 6), (True, 40)])
def test_stokes_nonlinear_residual_matches_host(CN, n_t):
    """ctl_stokes_nonlinear_residual after set_forward with per-level non-symmetric D_v_i (and D_p_i), on b lifted on
    the device, against the reference's residual: r to 1e-12 of its largest entry, constrained velocity rows exactly
    zero, the norm to 1e-12, b and x bit-unchanged, and the same bits on a second call."""
    import torch
    from control_b200.stokes import StokesSystem
    c = _ns_case(CN, n_t=n_t)
    q, N, bd = c["q"], c["N"], c["q"]["bdofs"]
    s = StokesSystem(q["M"], q["D_v"](np.zeros(c["n_v"]), 0.0), q["B"], q["sq"]["M_p"], q["sq"]["L_p"], n_t=n_t,
                     beta=q["beta"], CN=CN, time_interval=q["time_interval"], bc_dofs_v=bd,
                     D_p=q["D_p"](np.zeros(c["n_v"]), 0.0))
    s.set_forward(c["K_it"], c["P_it"])
    b = s.lift_bc_device(c["g"], s.to_device(*c["b_hom"]))
    x = s.to_device(c["x0"], c["x1"])
    b_keep, x_keep = b.clone(), x.clone()
    r = s.new_vector()
    norm = s.nonlinear_residual(b, x, r)
    r0, r1 = s.to_host_blocks(r)
    scale = max(np.abs(c["e0"]).max(), np.abs(c["e1"]).max())
    assert np.abs(r0 - c["e0"]).max() <= 1e-12 * scale
    assert np.abs(r1 - c["e1"]).max() <= 1e-12 * scale
    assert np.all(r0[:, bd] == 0.0)
    assert abs(norm - c["ref_norm"]) <= 1e-12 * c["ref_norm"]
    assert torch.equal(b, b_keep) and torch.equal(x, x_keep)
    r2 = s.new_vector()
    assert s.nonlinear_residual(b, x, r2) == norm and torch.equal(r, r2)
    assert np.array_equal(s.velocity_state_to_host(x), c["x0"][:N])
    s.close()


@pytest.mark.gpu
def test_stokes_nonlinear_residual_errors():
    """Null and aliased pointers return CTL_ERR_ARG with a message, a call with an unassembled handle CTL_ERR_STATE;
    wrong tensors raise ValueError in Python; the system stays usable."""
    import torch
    from control_b200 import _lib as L
    from control_b200.stokes import StokesSystem
    q = kat.reference_navier_stokes_problem(True, nx=2, n_t=3)
    s = StokesSystem(q["M"], q["D_v"](np.zeros(q["M"].shape[0]), 0.0), q["B"], q["sq"]["M_p"], q["sq"]["L_p"], n_t=3,
                     beta=q["beta"], CN=True, time_interval=q["time_interval"], bc_dofs_v=q["bdofs"])
    lib = L.load()
    b, x, r = s.new_vector(), s.new_vector(), s.new_vector()
    out = C.c_double()
    assert lib.ctl_stokes_nonlinear_residual(s._s, None, x.data_ptr(), r.data_ptr(), C.byref(out)) == -1
    assert b"null argument" in lib.ctl_last_error(s.velocity._h)
    assert lib.ctl_stokes_nonlinear_residual(s._s, b.data_ptr(), x.data_ptr(), r.data_ptr(), None) == -1
    assert lib.ctl_stokes_nonlinear_residual(s._s, b.data_ptr(), x.data_ptr(), b.data_ptr(), C.byref(out)) == -1
    assert b"alias" in lib.ctl_last_error(s.velocity._h)
    assert lib.ctl_stokes_nonlinear_residual(None, b.data_ptr(), x.data_ptr(), r.data_ptr(), C.byref(out)) == -1
    for bad in (torch.zeros(s.vec_len() - 1, dtype=torch.float64, device=s.device),
                torch.zeros(s.vec_len(), dtype=torch.float32, device=s.device),
                torch.zeros(2 * s.vec_len(), dtype=torch.float64, device=s.device)[::2],
                np.zeros(s.vec_len())):
        with pytest.raises(ValueError):
            s.nonlinear_residual(b, bad, r)
    data = q["M"].sorted_indices().data.copy()
    assert lib.ctl_set_values(s.velocity._h, L.CTL_MAT_M, -1, data.ctypes.data) == 0
    assert lib.ctl_stokes_nonlinear_residual(s._s, b.data_ptr(), x.data_ptr(), r.data_ptr(), C.byref(out)) == -3
    assert b"not assembled" in lib.ctl_last_error(s.velocity._h)
    assert lib.ctl_assemble(s.velocity._h) == 0
    assert s.nonlinear_residual(b, x, r) == 0.0
    s.close()


def _spy_host_residual(monkeypatch):
    from control_b200 import Control
    calls = []
    orig = Control.Instationary.non_linear_res_eval

    def spy(self, *a, **k):
        calls.append(1)
        return orig(self, *a, **k)
    monkeypatch.setattr(Control.Instationary, "non_linear_res_eval", spy)
    return calls


_NS_SP = {"linear_solver": "fgmres", "maximum_iterations": 200, "relative_tolerance": 1e-8, "absolute_tolerance": 0.0}


@pytest.mark.gpu
@pytest.mark.parametrize("CN", [True, False])
def test_navier_stokes_device_loop_matches_oracle(CN, monkeypatch):
    """incompressible_non_linear_solve(device_loop=True) on the lid-driven cavity (4 x 4 Q2-Q1 cells) against the
    oracle's loop with the same time-dependent lid data, with the tolerances of the host loop's GPU test; the host
    residual is never evaluated."""
    q = kat.reference_navier_stokes_problem(CN, nx=4, n_t=6)
    sq = q["sq"]
    calls = _spy_host_residual(monkeypatch)
    c, space_p = _ns_control(q)
    k = c.incompressible_non_linear_solve("constant", space_p=space_p, solver_parameters=dict(_NS_SP),
                                          lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"],
                                          print_error_non_linear=False, device_loop=True)
    assert not calls
    out = ostokes.incompressible_non_linear_solve(
        q["M"], q["D_v"], q["B"], sq["M_p"], sq["L_p"], q["D_p"], beta=q["beta"], n_t=q["n_t"], CN=CN,
        time_interval=q["time_interval"], bdofs_v=q["bdofs"], v_d=q["v_d"], f=q["f"], bc_values=q["bc_values"],
        solver_parameters=dict(_NS_SP), lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"])
    assert k == out["iterations"] and k >= 2
    assert np.allclose(c.non_linear_history, out["history"], rtol=1e-3)
    assert np.abs(c._v - out["v"]).max() < 1e-5 * np.abs(out["v"]).max()
    assert np.abs(c._zeta - out["zeta"]).max() < 1e-5 * np.abs(out["zeta"]).max()
    assert max(abs(a - b) for a, b in zip(c.inner_iterations, out["inner_its"])) <= 2
    assert np.all(c._v[:, q["bdofs"]] == q["bc_values"]) and np.all(c._zeta[:, q["bdofs"]] == 0.0)
    c.close()


@pytest.mark.gpu
def test_navier_stokes_device_loop_matches_host_loop():
    """The device and the host loop on the same problem and GPU: the increment solves see the same right-hand side up
    to rounding, so the outer iteration counts agree and the residual histories agree to 1e-6."""
    q = kat.reference_navier_stokes_problem(True, nx=4, n_t=6)
    runs = []
    for device_loop in (True, False):
        c, space_p = _ns_control(q)
        k = c.incompressible_non_linear_solve("constant", space_p=space_p, solver_parameters=dict(_NS_SP),
                                              lambda_v_bounds=q["lambda_v_bounds"],
                                              lambda_p_bounds=q["lambda_p_bounds"], print_error_non_linear=False,
                                              device_loop=device_loop)
        runs.append((k, list(c.non_linear_history), c._v.copy(), c._p.copy(), list(c.inner_iterations)))
        c.close()
    (kd, hd, vd, pd, itd), (kh, hh, vh, ph, ith) = runs
    assert kd == kh and kd >= 2
    assert np.allclose(hd, hh, rtol=1e-6)
    assert np.abs(vd - vh).max() <= 1e-6 * np.abs(vh).max()
    assert np.abs(pd - ph).max() <= 1e-6 * np.abs(ph).max()
    assert itd == ith


@pytest.mark.gpu
@pytest.mark.parametrize("CN,gauss_newton", [(True, False), (False, False), (True, True)])
def test_heat_device_loop_with_inhomogeneous_data_matches_oracle(CN, gauss_newton, monkeypatch):
    """non_linear_solve(device_loop=True) with time-dependent inhomogeneous Dirichlet data (non-linear diffusion)
    against ocontrol.non_linear_solve(bc_values=g); the host residual is never evaluated."""
    nx, n_t = 6, 5
    q = kat.heat_problem(nx, n_t, CN, beta=1e-2)
    Dv = fem.nonlinear_diffusion_p1_2d(nx, nx, 2.0, 2.0)
    xb, yb = q["coords"][q["bdofs"], 0], q["coords"][q["bdofs"], 1]
    g = 0.3 * np.stack([np.cos(xb + t) + 0.5 * yb for t in q["tau"] * np.arange(n_t)])
    sp_ = {"linear_solver": "fgmres", "maximum_iterations": 200, "relative_tolerance": 1e-7 if CN else 1e-6,
           "absolute_tolerance": 0.0, "gmres_restart": 100}
    calls = _spy_host_residual(monkeypatch)
    c = _heat_control(q, Dv, g, CN, gauss_newton)
    k = c.non_linear_solve(solver_parameters=dict(sp_), lambda_v_bounds=q["lambda_v_bounds"], max_non_linear_iter=6,
                           print_error_non_linear=False, device_loop=True)
    assert not calls
    ref = ocontrol.non_linear_solve(q["M"], lambda v, t: Dv(v, gauss_newton), beta=q["beta"], n_t=n_t, CN=CN,
                                    time_interval=q["time_interval"], bdofs=q["bdofs"], v_d=q["v_d"], f=q["f"],
                                    solver_parameters=dict(sp_), lambda_v_bounds=q["lambda_v_bounds"],
                                    max_non_linear_iter=6, bc_values=g)
    assert k == ref["iterations"] and k >= 2
    assert np.allclose(c.non_linear_history, ref["history"], rtol=1e-4)
    assert np.abs(c._v - ref["v"]).max() < 1e-5 * np.abs(ref["v"]).max()
    assert np.abs(c._zeta - ref["zeta"]).max() < 1e-5 * np.abs(ref["zeta"]).max()
    c.close()
