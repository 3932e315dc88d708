"""GPU parity of the instationary Stokes control path (operator, pressure-Schur preconditioner,
outer solve) against oracle/stokes.py, through the C ABI.  fp64; tolerances next to each
assertion.  Taylor-Hood P2-P1 on the unit square, zero Dirichlet velocity data."""
import numpy as np
import pytest
import torch

from oracle import stokes
from synthetic import fem

pytestmark = pytest.mark.gpu

LAMBDA_V = (0.3924, 2.0598)      # P2 vector mass matrix, measured on this mesh family (oracle/fem.py)
LAMBDA_P = (0.5, 2.0)            # P1 mass matrix (Wathen)
AMG = dict(coarse_max=40)
AMG_P = dict(coarse_max=20)


def _problem(nx, n_t, CN, beta=1e-2):
    th = fem.assemble_taylor_hood_2d(nx, nx, 1.0, 1.0)
    return dict(th=th, n_t=n_t, CN=CN, beta=beta, tau=1.0 / (n_t - 1.0), N=n_t - 1 if CN else n_t)


def _system(q):
    from control_b200.stokes import StokesSystem
    th = q["th"]
    return StokesSystem(th["M_v"], th["K_v"], th["B"], th["M_p"], th["K_p"], n_t=q["n_t"], beta=q["beta"], CN=q["CN"],
                        bc_dofs_v=th["bdofs_v"])


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


@pytest.mark.parametrize("CN,n_t", [(True, 2), (False, 2), (True, 5), (True, 9), (False, 5), (False, 8), (True, 33), (True, 70)])
def test_stokes_operator_matches_oracle(CN, n_t):
    q = _problem(5, n_t, CN)
    th, N = q["th"], q["N"]
    s = _system(q)
    rng = np.random.default_rng(n_t)
    x0 = rng.standard_normal((2 * N, s.n_v))
    x1 = rng.standard_normal((2 * N, s.n_p))
    y0, y1 = s.to_host_blocks(s.apply(s.to_device(x0, x1)))
    r0, r1 = stokes.stokes_apply_fused(th["M_v"], th["K_v"], th["B"], q["tau"], q["beta"], n_t, CN, th["bdofs_v"], x0, x1)
    assert _rel(y0, r0) < 1e-13          # same sums, different association
    assert _rel(y1, r1) < 1e-13
    assert s.kernel_launches() > 0
    s.close()


def _oracle_pc(q, **kw):
    th = q["th"]
    return stokes.construct_stokes_pc(th["M_v"], th["K_v"], th["B"], th["M_p"], th["K_p"], q["tau"], q["beta"], q["n_t"],
                                      q["CN"], th["bdofs_v"], lambda_v_bounds=LAMBDA_V, lambda_p_bounds=LAMBDA_P,
                                      inner="amg", amg_params=AMG, amg_params_p=AMG_P, **kw)


@pytest.mark.parametrize("CN", [True, False])
def test_stokes_pc_fn_matches_oracle(CN):
    q = _problem(6, 5, CN)
    th, N = q["th"], q["N"]
    s = _system(q)
    s.setup_preconditioner(lambda_v_bounds=LAMBDA_V, lambda_p_bounds=LAMBDA_P, amg=AMG, amg_p=AMG_P)
    rng = np.random.default_rng(3)
    b0 = rng.standard_normal((2 * N, s.n_v))
    b0[:, th["bdofs_v"]] = 0.0
    b1 = rng.standard_normal((2 * N, s.n_p))
    b1 -= b1.mean(axis=1, keepdims=True)
    u0, u1 = s.to_host_blocks(s.pc_apply(s.to_device(b0, b1), raw=True))
    r0, r1 = _oracle_pc(q)(b0, b1)
    # The five inner GMRES iterations run past convergence on this small mesh: the last Krylov
    # directions are normalised rounding noise, so pc_fn amplifies a 1e-15 relative perturbation
    # of b to ~1e-8 in u (measured on the oracle itself); 5e-7 bounds that, not the arithmetic.
    assert _rel(u0, r0) < 5e-7
    assert _rel(u1, r1) < 5e-7
    # Preconditioner.apply: the nullspace wrapping (general right-hand side)
    c0 = rng.standard_normal((2 * N, s.n_v))
    c1 = rng.standard_normal((2 * N, s.n_p))
    w0, w1 = s.to_host_blocks(s.pc_apply(s.to_device(c0, c1)))
    d0 = c0.copy()
    d0[:, th["bdofs_v"]] = 0.0
    d1 = c1 - c1.mean(axis=1, keepdims=True)
    e0, e1 = _oracle_pc(q)(d0, d1)
    e0 = e0.copy()
    e0[:, th["bdofs_v"]] = c0[:, th["bdofs_v"]]
    e1 = e1 - e1.mean(axis=1, keepdims=True) + c1.mean(axis=1, keepdims=True)
    assert _rel(w0, e0) < 5e-7
    assert _rel(w1, e1) < 5e-7
    s.close()


@pytest.mark.parametrize("CN", [True, False])
def test_stokes_solve_matches_oracle(CN):
    q = _problem(6, 5, CN)
    th, N = q["th"], q["N"]
    s = _system(q)
    s.setup_preconditioner(lambda_v_bounds=LAMBDA_V, lambda_p_bounds=LAMBDA_P, amg=AMG, amg_p=AMG_P)
    rng = np.random.default_rng(7)
    xr0 = rng.standard_normal((2 * N, s.n_v))
    xr0[:, th["bdofs_v"]] = 0.0
    xr1 = rng.standard_normal((2 * N, s.n_p))
    xr1 -= xr1.mean(axis=1, keepdims=True)
    b0, b1 = stokes.stokes_apply_fused(th["M_v"], th["K_v"], th["B"], q["tau"], q["beta"], q["n_t"], CN, th["bdofs_v"],
                                       xr0, xr1)
    sp_ = {"linear_solver": "fgmres", "maximum_iterations": 300, "relative_tolerance": 1e-8 if CN else 1e-6,
           "absolute_tolerance": 0.0, "gmres_restart": 100}
    u0 = np.zeros_like(xr0)
    u1 = np.zeros_like(xr1)
    info = s.solve(u0, u1, b0, b1, solver_parameters=sp_)
    o0, o1, res = stokes.stokes_solve(th["M_v"], th["K_v"], th["B"], th["M_p"], th["K_p"], beta=q["beta"], n_t=q["n_t"], CN=CN,
                                      bdofs_v=th["bdofs_v"], b_0=b0, b_1=b1, solver_parameters=sp_, pc_fn=_oracle_pc(q))
    assert info.reason == res.reason > 0
    if CN:
        assert abs(info.its - res.its) <= 1
        k = min(len(info.history), len(res.history), 10)
        assert np.allclose(info.history[:k], res.history[:k], rtol=1e-4)     # see the pc_fn test for the sensitivity
        assert _rel(u0, o0) < 1e-5 and _rel(u0, xr0) < 1e-4        # solver tolerance times the conditioning
        assert _rel(u1, o1) < 1e-3
    else:
        # BE: after a fast first phase the residual creeps (the epsilon-regularised last block), and in
        # that phase the iteration is rounding dominated: on this right-hand side the preconditioner maps
        # differences of 1e-13 (AMG Galerkin products) to 5e-6, and the two runs need 32 (GPU) and 116
        # (oracle) iterations with identical leading histories.  Compare what is well defined: the first
        # residuals, convergence, and the true residual of the returned solution.
        assert np.allclose(info.history[:5], res.history[:5], rtol=1e-3)
        r0, r1 = stokes.stokes_apply_fused(th["M_v"], th["K_v"], th["B"], q["tau"], q["beta"], q["n_t"], CN, th["bdofs_v"],
                                           u0, u1)
        bnorm = np.sqrt((b0 ** 2).sum() + (b1 ** 2).sum())
        assert np.sqrt(((b0 - r0) ** 2).sum() + ((b1 - r1) ** 2).sum()) < 1e-5 * bnorm      # rtol 1e-6, CGS drift
    assert info.n_pc >= info.its
    s.close()


def test_stokes_user_preconditioner_hook(capsys):
    """``P=`` of ``incompressible_linear_solve`` (control/control.py:3592-3594, 4686-4689): a user callable
    ``pc_fn(u_0, u_1, b_0, b_1)`` on the blocks of the outer system, called through ctl_stokes_set_pc_callback.  Handing
    the in-built preconditioner back in as the user's P must reproduce the in-built solve (same count, same solution);
    the callable sees projected right-hand sides (Dirichlet rows zero, pressure blocks mean free) and zero u's; an
    exception inside it surfaces as the reference's RuntimeError, and the next solve starts afresh.  The solve prints
    its residual history exactly when ``monitor_convergence`` is set."""
    q = _problem(6, 5, True)
    th, N = q["th"], q["N"]
    s = _system(q)
    s.setup_preconditioner(lambda_v_bounds=LAMBDA_V, lambda_p_bounds=LAMBDA_P, amg=AMG, amg_p=AMG_P)
    rng = np.random.default_rng(7)
    xr0 = rng.standard_normal((2 * N, s.n_v))
    xr0[:, th["bdofs_v"]] = 0.0
    xr1 = rng.standard_normal((2 * N, s.n_p))
    xr1 -= xr1.mean(axis=1, keepdims=True)
    b0, b1 = stokes.stokes_apply_fused(th["M_v"], th["K_v"], th["B"], q["tau"], q["beta"], q["n_t"], True, th["bdofs_v"],
                                       xr0, xr1)
    sp_ = {"linear_solver": "fgmres", "maximum_iterations": 300, "relative_tolerance": 1e-8, "absolute_tolerance": 0.0,
           "gmres_restart": 100}
    u0, u1 = np.zeros_like(xr0), np.zeros_like(xr1)
    ref = s.solve(u0, u1, b0, b1, solver_parameters=sp_)
    inner = s.builtin_pc_fn()
    seen = []

    def P(w_0, w_1, c_0, c_1):
        assert not w_0.any() and not w_1.any()
        assert not c_0[:, th["bdofs_v"]].any() and np.abs(c_1.mean(axis=1)).max() <= 1e-12 * max(np.abs(c_1).max(), 1e-300)
        seen.append(1)
        inner(w_0, w_1, c_0, c_1)
    w0, w1 = np.zeros_like(xr0), np.zeros_like(xr1)
    info = s.solve(w0, w1, b0, b1, solver_parameters=sp_, pc_fn=P)
    assert info.reason > 0 and len(seen) == info.n_pc >= info.its
    assert abs(info.its - ref.its) <= 1
    assert _rel(w0, u0) < 1e-6 and _rel(w1, u1) < 1e-4

    def broken(w_0, w_1, c_0, c_1):
        raise ValueError("user preconditioner failed")
    with pytest.raises(Exception):
        s.solve(np.zeros_like(xr0), np.zeros_like(xr1), b0, b1, solver_parameters=sp_, pc_fn=broken)
    capsys.readouterr()
    info = s.solve(np.zeros_like(xr0), np.zeros_like(xr1), b0, b1, solver_parameters=dict(sp_, monitor_convergence=False))
    assert info.reason > 0 and abs(info.its - ref.its) <= 1
    assert capsys.readouterr().out == ""
    info = s.solve(np.zeros_like(xr0), np.zeros_like(xr1), b0, b1, solver_parameters=dict(sp_, monitor_convergence=True))
    assert len(info.history) > 1 and capsys.readouterr().out.splitlines() == \
        [f"KSP: iteration {it:d}, residual norm {r:.16e}" for it, r in enumerate(info.history)]
    s.close()


def test_stokes_rejects_mismatched_handles():
    from control_b200 import CtlError, MultiBlockSystem
    from control_b200 import _lib as L
    import ctypes as C
    th = fem.assemble_taylor_hood_2d(3, 3, 1.0, 1.0)
    a = MultiBlockSystem(th["M_v"], th["K_v"], n_t=5, beta=1e-2, CN=True, bc_dofs=th["bdofs_v"])
    b = MultiBlockSystem(th["M_p"], th["K_p"], n_t=6, beta=1e-2, CN=True, stream=a.stream)
    B = th["B"].tocsr()
    ip, ix = B.indptr.astype(np.int32), B.indices.astype(np.int32)
    out = C.c_void_p()
    rc = a._lib.ctl_stokes_create(a._h, b._h, ip.ctypes.data, ix.ctypes.data, B.data.ctypes.data, C.byref(out))
    assert rc == -1 and b"share" in a._lib.ctl_last_error(a._h)
    with pytest.raises(CtlError):
        L.check(a._h, rc)
    a.close()
    b.close()


@pytest.mark.parametrize("CN", [True, False])
def test_control_incompressible_linear_solve_matches_oracle(CN):
    """The caller of the Stokes path: Control.Instationary.incompressible_linear_solve
    (control/control.py:3592-4725) on assembled objects, against the oracle's restatement."""
    import kat
    from control_b200 import Control
    q = kat.stokes_problem(6, 6, CN)
    th = q["th"]
    times = q["tau"] * np.arange(q["n_t"])
    lookup = {round(float(t), 12): i for i, t in enumerate(times)}
    c = Control.Instationary(q["M"], q["K"], desired_state=lambda t: (q["v_d"][lookup[round(float(t), 12)]],
                                                                    q["v_hat"][lookup[round(float(t), 12)]]),
                             force_f=lambda t: q["f"][lookup[round(float(t), 12)]], beta=q["beta"], CN=CN, n_t=q["n_t"],
                             time_interval=q["time_interval"], bc_dofs=q["bdofs"])
    sp_ = {"linear_solver": "fgmres", "maximum_iterations": 200, "relative_tolerance": 1e-8, "absolute_tolerance": 0.0,
           "gmres_restart": 100}
    info = c.incompressible_linear_solve("constant", space_p=dict(B=th["B"], M_p=th["M_p"], K_p=th["K_p"]),
                                         solver_parameters=sp_, lambda_v_bounds=q["lambda_v_bounds"],
                                         lambda_p_bounds=q["lambda_p_bounds"], amg=AMG, amg_p=AMG_P)
    v, zeta, p, mu, res = stokes.incompressible_linear_solve(
        th["M_v"], th["K_v"], th["B"], th["M_p"], th["K_p"], beta=q["beta"], n_t=q["n_t"], CN=CN,
        time_interval=q["time_interval"], bdofs_v=q["bdofs"], v_d=q["v_d"], f=q["f"], solver_parameters=sp_,
        lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"], amg_params=AMG, amg_params_p=AMG_P)
    assert info.reason == res.reason > 0
    assert abs(info.its - res.its) <= max(1, int(0.03 * res.its))
    assert _rel(c._v, v) < 1e-5 and _rel(c._zeta, zeta) < 1e-5        # solver tolerance 1e-8 x conditioning
    assert _rel(c._p, p) < 1e-4 and _rel(c._mu, mu) < 1e-4
    # the computed state is discretely divergence free (the constraint rows of the KKT system)
    div = (th["B"] @ c._v[1:].T).T
    div -= div.mean(axis=1, keepdims=True)
    assert np.abs(div).max() < 1e-6 * np.abs(th["B"]).sum(axis=1).max() * np.abs(c._v).max()
    c.close()


@pytest.mark.parametrize("CN", [True, False])
def test_instationary_stokes_known_answer_on_gpu(CN):
    """The reference-style known-answer problem (tests/kat.py::instationary_stokes_kat: right-hand
    sides built row by row from the block stencils, analytic v / zeta / p / mu) through the CUDA path:
    Control.Instationary.incompressible_linear_solve with ready blocks (v_d=, f=, div_v=, div_zeta=)."""
    import kat
    from control_b200 import Control
    q = kat.instationary_stokes_kat(CN)
    sq = q["sq"]
    c = Control.Instationary(q["M"], q["K"], beta=q["beta"], CN=CN, n_t=q["n_t"], time_interval=(0.0, 1.0),
                             bc_dofs=q["bdofs"])
    info = c.incompressible_linear_solve("constant", space_p=dict(B=q["B"], M_p=sq["M_p"], K_p=sq["L_p"]),
                                         solver_parameters=q["solver_parameters"], v_d=q["v_d"], f=q["f"],
                                         div_v=q["div_v"], div_zeta=q["div_zeta"],
                                         lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"])
    assert info.reason > 0
    v_u = c._v[1:] if CN else c._v
    z_u = c._zeta[:-1] if CN else c._zeta
    scale = kat.l2_error(q["M"], q["v_unknown"], 0 * q["v_unknown"])
    assert kat.l2_error(q["M"], v_u, q["v_unknown"]) < 1e-9 * scale        # solver tolerance 1e-13 x conditioning
    assert kat.l2_error(q["M"], z_u, q["z_unknown"]) < 1e-9 * scale
    Mp = sq["M_p"]

    def shift(a):
        return a - (a @ (Mp @ np.ones(Mp.shape[0])))[:, None]
    pscale = kat.l2_error(Mp, shift(q["p_ref"]), 0 * q["p_ref"])
    assert kat.l2_error(Mp, shift(c._p), shift(q["p_ref"])) < 1e-8 * pscale
    assert kat.l2_error(Mp, shift(c._mu), shift(q["mu_ref"])) < 1e-8 * pscale
    c.close()


@pytest.mark.parametrize("CN", [True, False])
def test_stokes_control_with_inhomogeneous_velocity_data(CN):
    """Time-dependent inhomogeneous Dirichlet velocity data (the setting of the reference's own
    instationary Stokes tests, test/test_control.py:3045-3302) through the CUDA path against the oracle,
    whose lifting is checked against a direct un-eliminated solve in tests/test_oracle.py."""
    import kat
    from control_b200 import Control
    q = kat.stokes_problem(5, 5, CN)
    th, bd = q["th"], q["bdofs"]
    n_v = q["M"].shape[0]
    comp = (bd % 2 == 0)

    def bc_values(t):
        return (1.0 + t) * np.where(comp, 1.0, 0.5)          # a constant vector field: zero net flux
    times = q["tau"] * np.arange(q["n_t"])
    g = np.stack([bc_values(t) for t in times])
    v_0 = np.zeros(n_v)
    v_0[0::2], v_0[1::2] = 1.0, 0.5
    idx = {round(float(t), 12): i for i, t in enumerate(times)}
    c = Control.Instationary(q["M"], q["K"], desired_state=lambda t: (q["v_d"][idx[round(float(t), 12)]],
                                                                    q["v_hat"][idx[round(float(t), 12)]]),
                             force_f=lambda t: q["f"][idx[round(float(t), 12)]], beta=q["beta"], CN=CN, n_t=q["n_t"],
                             time_interval=q["time_interval"], bc_dofs=bd, bc_values=bc_values, initial_condition=v_0)
    sp_ = {"linear_solver": "fgmres", "maximum_iterations": 300, "relative_tolerance": 1e-9, "absolute_tolerance": 0.0,
           "gmres_restart": 100}
    info = c.incompressible_linear_solve("constant", space_p=dict(B=th["B"], M_p=th["M_p"], K_p=th["K_p"]),
                                         solver_parameters=sp_, lambda_v_bounds=q["lambda_v_bounds"],
                                         lambda_p_bounds=q["lambda_p_bounds"], amg=AMG, amg_p=AMG_P)
    v, zeta, p, mu, res = stokes.incompressible_linear_solve(
        th["M_v"], th["K_v"], th["B"], th["M_p"], th["K_p"], beta=q["beta"], n_t=q["n_t"], CN=CN,
        time_interval=q["time_interval"], bdofs_v=bd, v_d=q["v_d"], f=q["f"], v_0=v_0, bc_values=g,
        solver_parameters=sp_, lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"],
        amg_params=AMG, amg_params_p=AMG_P)
    assert info.reason == res.reason > 0
    assert abs(info.its - res.its) <= max(1, int(0.03 * res.its))
    assert _rel(c._v, v) < 1e-5 and _rel(c._zeta, zeta) < 1e-5
    assert _rel(c._p, p) < 1e-4 and _rel(c._mu, mu) < 1e-4
    assert np.array_equal(c._v[1:][:, bd], g[1:])
    c.close()


@pytest.mark.parametrize("CN", [False, True])
def test_reference_instationary_stokes_exact_solution_problem_on_gpu(CN):
    """The reference's two instationary Stokes tests (test/test_control.py:3045-3302) through the CUDA
    path with the reference's default solver parameters: converges, matches the oracle, and reproduces
    the analytic velocity up to the discretisation error."""
    import kat
    from control_b200 import Control
    q = kat.reference_stokes_exact_problem(CN)
    sq, bd = q["sq"], q["bdofs"]
    times = q["tau"] * np.arange(q["n_t"])
    idx = {round(float(t), 12): i for i, t in enumerate(times)}
    c = Control.Instationary(q["M"], q["K"], desired_state=lambda t: (q["v_d"][idx[round(float(t), 12)]],
                                                                    q["v_hat"][idx[round(float(t), 12)]]),
                             force_f=lambda t: q["f"][idx[round(float(t), 12)]], beta=q["beta"], CN=CN, n_t=q["n_t"],
                             time_interval=q["time_interval"], bc_dofs=bd,
                             bc_values=lambda t: q["bc_values"][idx[round(float(t), 12)]], initial_condition=q["v_0"])
    info = c.incompressible_linear_solve("constant", space_p=dict(B=q["B"], M_p=sq["M_p"], K_p=sq["L_p"]),
                                         lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"],
                                         print_error=False)
    assert info.reason > 0 and info.its <= 40
    err = kat.l2_error(q["M"], c._v, q["true_v"]) / kat.l2_error(q["M"], q["true_v"], 0 * q["true_v"])
    assert err < (1e-4 if CN else 1e-3)
    v, zeta, p, mu, res = stokes.incompressible_linear_solve(
        q["M"], q["K"], q["B"], sq["M_p"], sq["L_p"], beta=q["beta"], n_t=q["n_t"], CN=CN,
        time_interval=q["time_interval"], bdofs_v=bd, v_d=q["v_d"], f=q["f"], v_0=q["v_0"],
        bc_values=q["bc_values"], lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"])
    assert abs(info.its - res.its) <= 1
    assert _rel(c._v, v) < 1e-4          # both stop at rtol 1e-6
    c.close()
