"""Lifting of inhomogeneous, time-dependent Dirichlet data on the device (ctl_lift_bc, ctl_stokes_lift_bc).

CPU: the lifting of the host right-hand side is additive and equals an independent restatement, and the residual of
the outer Picard / Gauss-Newton loop with such data is the lifted right-hand side (K_i at the iterate) minus the
operator.  GPU: the device lifting against the host one, a linear solve and the device-resident non-linear loop
built on it against the oracle, the Stokes variant, and the argument / state errors."""
import numpy as np
import pytest
import scipy.sparse as sp

import kat
from oracle import control as ocontrol
from oracle import kkt
from synthetic import fem

SEED = 20261020


def _T(L0, L1, CN):
    return (kkt.apply_T_1(L0), kkt.apply_T_2(L1)) if CN else (L0, L1)


def _lift_restated(M, K_levels, tau, n_t, CN, bd, g):
    """-T L(g) from the time-coupling coefficients: L_0 = C_0 (M_bd g), L_1 = C_1 (M_bd g) + D_1 (K_bd g), the
    constrained rows zeroed, then T -- an independent restatement of the lift branch of build_rhs."""
    N = n_t - 1 if CN else n_t
    Mg = np.stack([M[:, bd] @ g[l] for l in range(n_t)])                   # (n_t, n)
    Kg = np.stack([K_levels[l][:, bd] @ g[l] for l in range(n_t)])
    C0, C1, D1 = np.zeros((N, n_t)), np.zeros((N, n_t)), np.zeros((N, n_t))
    for i in range(N):
        if CN:
            h = 0.5 * tau
            C0[i, i + 1] = h
            C1[i, i + 1] = 1.0
            D1[i, i + 1] = h
            if i > 0:
                C0[i, i] = h
                C1[i, i] = -1.0
                D1[i, i] = h
        else:
            if i < n_t - 1:
                C0[i, i] = tau
            C1[i, i] = 1.0
            D1[i, i] = tau
            if i > 0:
                C1[i, i - 1] = -1.0
    L0, L1 = C0 @ Mg, C1 @ Mg + D1 @ Kg
    L0[:, bd] = 0.0
    L1[:, bd] = 0.0
    T0, T1 = _T(L0, L1, CN)
    return -T0, -T1


def _per_level(K, n_t, rng):
    """n_t non-symmetric matrices on K's pattern."""
    out = []
    for _ in range(n_t):
        Ki = K.tocsr().copy()
        Ki.data = Ki.data * (1.0 + 0.2 * rng.standard_normal(Ki.data.size))
        out.append(Ki)
    return out


def _boundary_data(q, n_t, seed=0):
    xb, yb = q["coords"][q["bdofs"], 0], q["coords"][q["bdofs"], 1]
    times = q["tau"] * np.arange(n_t)
    return 0.3 * np.stack([np.cos(xb + t + seed) + 0.5 * yb for t in times])


# ---------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("CN", [True, False])
@pytest.mark.parametrize("per_level", [False, True])
def test_host_lifting_is_additive_and_matches_restatement(CN, per_level):
    from control_b200.control import build_rhs
    rng = np.random.default_rng(SEED)
    n_t = 6
    q = kat.heat_problem(7, n_t, CN, beta=1e-2)
    M, K, tau = q["M"], q["K"], q["tau"]
    bd = rng.permutation(q["bdofs"]).astype(np.int32)                          # unsorted list
    assert not np.all(np.diff(bd) > 0)
    Kl = _per_level(K, n_t, rng) if per_level else [K] * n_t
    g = rng.standard_normal((n_t, bd.size))
    v_0 = rng.standard_normal(M.shape[0])
    args = (M, Kl[0], tau, n_t, CN, bd, q["v_d"], q["f"], v_0)
    with_g = build_rhs(*args, bc_values=g, K_levels=Kl if per_level else None)
    without = build_rhs(*args, K_levels=Kl if per_level else None)
    ref = _lift_restated(M, Kl, tau, n_t, CN, bd, g)
    for a, b, r in zip(with_g, without, ref):
        assert np.abs((a - b) - r).max() <= 1e-14 * max(np.abs(r).max(), 1.0)
        assert np.all(r[:, bd] == 0.0)


@pytest.mark.parametrize("CN,gauss_newton", [(True, False), (False, False), (True, True), (False, True)])
def test_non_linear_residual_with_inhomogeneous_data_is_lifted_rhs_minus_operator(CN, gauss_newton):
    """oracle non_linear_res_eval at an iterate that carries g on the constrained dofs (as non_linear_solve with
    bc_values leaves it) == T^-1 (b - A x), b = the homogeneous right-hand side lifted with K_i at the iterate.  For
    CN the initial condition in b is level 0 of the iterate (non_linear_solve re-imposes g_0 there as well)."""
    from control_b200.control import build_rhs
    rng = np.random.default_rng(SEED + 1)
    nx, n_t = 6, 5
    q = kat.heat_problem(nx, n_t, CN, beta=1e-2)
    M, tau, bd, beta = q["M"], q["tau"], q["bdofs"], q["beta"]
    Dv = fem.nonlinear_diffusion_p1_2d(nx, nx, 2.0, 2.0)
    times = tau * np.arange(n_t)
    n = M.shape[0]
    g = _boundary_data(q, n_t)
    v_old = rng.standard_normal((n_t, n))
    v_old[:, bd] = g
    zeta_old = rng.standard_normal((n_t, n))
    zeta_old[:, bd] = 0.0
    v_0 = rng.standard_normal(n)
    if CN:
        zeta_old[-1] = 0.0
        v_0 = v_old[0].copy()

    def D(v, t):
        return Dv(v, gauss_newton)
    r0, r1 = ocontrol.non_linear_res_eval(M, D, times, tau, beta, n_t, CN, bd, v_old, zeta_old, v_0, q["v_d"], q["f"])
    K_it = [D(v_old[i], times[i]) for i in range(n_t)]
    # homogeneous right-hand side: the initial-condition terms carry D_v(v_0) (control.py:3000-3004, 3217-3240)
    b0, b1 = build_rhs(M, D(v_0, times[0]), tau, n_t, CN, bd, q["v_d"], q["f"], v_0)
    l0, l1 = _lift_restated(M, K_it, tau, n_t, CN, bd, g)
    x0, x1 = (v_old[1:], zeta_old[:-1]) if CN else (v_old, zeta_old)
    y0, y1 = kkt.kkt_apply_fused(M, K_it, tau, beta, n_t, CN, bd, x0, x1)
    e0, e1 = _T(r0, r1, CN)
    d0, d1 = b0 + l0 - y0, b1 + l1 - y1
    d0[:, bd] = 0.0
    d1[:, bd] = 0.0
    scale = max(np.abs(e0).max(), np.abs(e1).max())
    assert np.abs(d0 - e0).max() <= 1e-12 * scale and np.abs(d1 - e1).max() <= 1e-12 * scale


# ---------------------------------------------------------------------------------------------------------- GPU
def _host_lift(M, K, tau, n_t, CN, bd, g, K_levels=None):
    """build_rhs(bc_values=g) - build_rhs(bc_values=None) on zero data."""
    from control_b200.control import build_rhs
    n = M.shape[0]
    z = np.zeros((n_t, n))
    args = (M, K, tau, n_t, CN, bd, z, z, np.zeros(n))
    a = build_rhs(*args, bc_values=g, K_levels=K_levels)
    b = build_rhs(*args, K_levels=K_levels)
    return a[0] - b[0], a[1] - b[1]


@pytest.mark.gpu
@pytest.mark.parametrize("CN", [True, False])
@pytest.mark.parametrize("per_level", [False, True])
@pytest.mark.parametrize("layout", ["block_major", "time_fastest"])
def test_device_lifting_matches_host(CN, per_level, layout):
    import torch
    from control_b200 import MultiBlockSystem
    from control_b200 import _lib as L
    rng = np.random.default_rng(SEED + 2)
    nx, n_t = 12, 7
    q = kat.heat_problem(nx, n_t, CN, beta=1e-2)
    M, tau = q["M"], q["tau"]
    bd = rng.permutation(q["bdofs"]).astype(np.int32)
    Dv = fem.nonlinear_diffusion_p1_2d(nx, nx, 2.0, 2.0)
    lay = {"block_major": L.CTL_LAYOUT_BLOCK_MAJOR, "time_fastest": L.CTL_LAYOUT_TIME_FASTEST}[layout]

    def K_of(v):               # Gauss-Newton values at an iterate: per level, non-symmetric
        return [Dv(v[i], True) for i in range(n_t)] if per_level else q["K"]
    v = rng.standard_normal((n_t, M.shape[0]))
    s = MultiBlockSystem(M, K_of(v), n_t=n_t, beta=q["beta"], CN=CN, time_interval=q["time_interval"], bc_dofs=bd)
    for rep in range(2):       # the second pass after set_K with new values: the boundary-column CSR is rebuilt
        if rep == 1:
            v = 2.0 * rng.standard_normal(v.shape)
            s.set_K(K_of(v))
        Kh = K_of(v)
        g = rng.standard_normal((n_t, bd.size))
        l0, l1 = _host_lift(M, Kh[0] if per_level else Kh, tau, n_t, CN, bd, g, K_levels=Kh if per_level else None)
        b0, b1 = rng.standard_normal((2, s.N, M.shape[0]))
        b_bm = s.to_device(b0, b1)
        b = s.convert(b_bm, L.CTL_LAYOUT_BLOCK_MAJOR, lay)
        before = b.clone()
        g_arg = torch.from_numpy(g).to(s.device) if rep == 1 else g            # host array and CUDA tensor
        s.lift_bc_device(g_arg, b, layout=lay)
        if lay == L.CTL_LAYOUT_TIME_FASTEST:                                   # padding columns stay zero
            pad = b.view(2, s.n_local, s.ld)[:, :, s.N:]
            assert torch.equal(pad, before.view(2, s.n_local, s.ld)[:, :, s.N:])
            b = s.convert(b, lay, L.CTL_LAYOUT_BLOCK_MAJOR)
        c0, c1 = s.to_host_blocks(b)
        scale = max(np.abs(l0).max(), np.abs(l1).max())
        assert np.abs((c0 - b0) - l0).max() <= 1e-13 * scale
        assert np.abs((c1 - b1) - l1).max() <= 1e-13 * scale
        assert np.array_equal(c0[:, bd], b0[:, bd]) and np.array_equal(c1[:, bd], b1[:, bd])   # bit-unchanged
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("CN", [True, False])
def test_linear_solve_from_lifted_device_rhs_matches_oracle(CN):
    """build_rhs_device(..., bc_values=g) on the manufactured heat problem of the reference's convergence studies
    (Dirichlet data 1, initial condition v(0)), solved on the device, against ocontrol.linear_solve(bc_values=g)."""
    import torch
    from control_b200 import MultiBlockSystem
    q = kat.mms_heat_problem(8, 12, CN)
    M, K, bd, n_t = q["M"], q["K"], q["bdofs"], q["n_t"]
    g = q["bc_values"] * (1.0 + 0.5 * np.sin(q["tau"] * np.arange(n_t)))[:, None]      # time dependent
    v_0 = q["v_0"].copy()
    v_0[bd] = g[0]
    # BE: below ~1e-8 the iteration sits on the rounding floor of classical Gram-Schmidt (DESIGN.md)
    sp_ = {"linear_solver": "fgmres", "maximum_iterations": 300, "relative_tolerance": 1e-11 if CN else 1e-7,
           "absolute_tolerance": 0.0, "gmres_restart": 100}
    ref = ocontrol.linear_solve(M, K, beta=q["beta"], n_t=n_t, CN=CN, time_interval=q["time_interval"], bdofs=bd,
                                v_d=q["v_d"], f=q["f"], v_0=v_0, bc_values=g, solver_parameters=sp_,
                                lambda_v_bounds=(0.5, 2.0), amg_params=dict(coarse_max=60))
    s = MultiBlockSystem(M, K, n_t=n_t, beta=q["beta"], CN=CN, time_interval=q["time_interval"], bc_dofs=bd)
    zero = torch.zeros(n_t * M.shape[0], dtype=torch.float64, device=s.device)
    b = s.build_rhs_device(torch.from_numpy(q["v_hat"]).to(s.device).reshape(-1), zero, v_0, bc_values=g)
    h0, h1 = s.to_host_blocks(b)
    scale = max(np.abs(ref["b_0"]).max(), np.abs(ref["b_1"]).max())
    assert np.abs(h0 - ref["b_0"]).max() <= 1e-13 * scale and np.abs(h1 - ref["b_1"]).max() <= 1e-13 * scale
    s.setup_preconditioner(lambda_v_bounds=(0.5, 2.0), coarse_max=60)
    u = s.new_vector()
    info = s.solve_device(b, u, solver_parameters=sp_)
    assert info.reason == ref["ksp"].reason > 0 and abs(info.its - ref["ksp"].its) <= 1
    u0, u1 = s.to_host_blocks(u)
    tol = 1e-7 if CN else 1e-4
    assert np.abs(u0 - ref["v_blocks"]).max() < tol * np.abs(ref["v_blocks"]).max()
    assert np.abs(u1 - ref["zeta_blocks"]).max() < tol * np.abs(ref["zeta_blocks"]).max()
    assert s.residual_norm(b, u) <= 1e-6 * float(b.norm())
    s.close()


def _device_non_linear_loop(q, Dv, g, CN, gauss_newton, sp_, max_it, rel_tol=1e-5, abs_tol=1e-8):
    """The device-resident Picard / Gauss-Newton loop of INTEGRATION.md section 6a with inhomogeneous data, step for
    step the loop of control/control.py:3377-3525: b is built once (homogeneous), every outer iteration after set_K
    copies it, lifts g with the K_i of the iterate, and takes the residual; g is written back into the iterate."""
    from control_b200 import MultiBlockSystem
    from control_b200.control import build_rhs
    M, tau, bd, n_t = q["M"], q["tau"], q["bdofs"], q["n_t"]
    n = M.shape[0]
    times = q["time_interval"][0] + tau * np.arange(n_t)

    def D(v, t):
        return Dv(v, gauss_newton)
    v_0 = np.zeros(n)
    v_old, zeta_old = np.zeros((n_t, n)), np.zeros((n_t, n))
    if CN:
        v_old[0] = v_0
    # the first residual sees the iterate before g is imposed; from then on level 0 carries g_0 as well (CN)
    v_0g = v_0.copy()
    if CN:
        v_0g[bd] = g[0]
    b_first = build_rhs(M, D(v_0, times[0]), tau, n_t, CN, bd, q["v_d"], q["f"], v_0)
    b_hom = build_rhs(M, D(v_0g, times[0]), tau, n_t, CN, bd, q["v_d"], q["f"], v_0g)
    s = MultiBlockSystem(M, [D(v_old[i], times[i]) for i in range(n_t)], n_t=n_t, beta=q["beta"], CN=CN,
                         time_interval=q["time_interval"], bc_dofs=bd)
    b_first_dev, b_hom_dev = s.to_device(*b_first), s.to_device(*b_hom)
    x = s.to_device(*((v_old[1:], zeta_old[:-1]) if CN else (v_old, zeta_old)))
    r = s.new_vector()
    history = [s.nonlinear_residual(b_first_dev, x, r)]
    k = 0
    while history[-1] > rel_tol * history[0] and history[-1] > abs_tol:
        s.setup_preconditioner(lambda_v_bounds=q["lambda_v_bounds"])
        d = s.new_vector()
        info = s.solve_device(r, d, solver_parameters=sp_)
        assert info.reason > 0
        x += d
        v_blocks = s.to_host_blocks(x)[0]
        if CN:
            v_old[1:] = v_blocks
        else:
            v_old = v_blocks.copy()
        v_old[:, bd] = g                                                    # control.py:3480-3483
        s.set_K([D(v_old[i], times[i]) for i in range(n_t)])
        b = b_hom_dev.clone()
        s.lift_bc_device(g, b)
        history.append(s.nonlinear_residual(b, x, r))
        k += 1
        if k + 1 > max_it:
            break
    x0, x1 = s.to_host_blocks(x)
    if CN:
        v_old[1:], zeta_old[:-1] = x0, x1
    else:
        v_old, zeta_old = x0.copy(), x1.copy()
    v_old[:, bd] = g
    zeta_old[:, bd] = 0.0
    s.close()
    return dict(v=v_old, zeta=zeta_old, history=history, iterations=k)


@pytest.mark.gpu
@pytest.mark.parametrize("CN,gauss_newton", [(True, False), (False, False), (True, True)])
def test_device_resident_non_linear_loop_with_inhomogeneous_data_matches_oracle(CN, gauss_newton):
    """Non-linear diffusion (BASELINE config C5 in small) with time-dependent inhomogeneous Dirichlet data: the
    device-resident loop against ocontrol.non_linear_solve(bc_values=g)."""
    nx, n_t = 6, 5
    q = kat.heat_problem(nx, n_t, CN, beta=1e-2)
    Dv = fem.nonlinear_diffusion_p1_2d(nx, nx, 2.0, 2.0)
    g = _boundary_data(q, n_t)
    sp_ = {"linear_solver": "fgmres", "maximum_iterations": 200, "relative_tolerance": 1e-7 if CN else 1e-6,
           "absolute_tolerance": 0.0, "gmres_restart": 100}
    out = _device_non_linear_loop(q, Dv, g, CN, gauss_newton, sp_, max_it=6)
    ref = ocontrol.non_linear_solve(q["M"], lambda v, t: Dv(v, gauss_newton), beta=q["beta"], n_t=n_t, CN=CN,
                                    time_interval=q["time_interval"], bdofs=q["bdofs"], v_d=q["v_d"], f=q["f"],
                                    solver_parameters=sp_, lambda_v_bounds=q["lambda_v_bounds"], max_non_linear_iter=6,
                                    bc_values=g)
    assert out["iterations"] == ref["iterations"] and out["iterations"] >= 2
    assert np.allclose(out["history"], ref["history"], rtol=1e-4)
    assert np.abs(out["v"] - ref["v"]).max() < 1e-5 * np.abs(ref["v"]).max()
    assert np.abs(out["zeta"] - ref["zeta"]).max() < 1e-5 * np.abs(ref["zeta"]).max()


@pytest.mark.gpu
@pytest.mark.parametrize("CN", [True, False])
def test_stokes_device_lifting_and_solve(CN):
    """ctl_stokes_lift_bc against the host lifting of incompressible_linear_solve (velocity and divergence rows) on
    the reference's instationary Stokes problem with an exact solution; then one outer solve from the lifted
    device vector recovers the analytic velocity."""
    import torch
    from control_b200.stokes import StokesSystem
    q = kat.reference_stokes_exact_problem(CN)
    sq, bd, n_t, tau = q["sq"], q["bdofs"], q["n_t"], q["tau"]
    M, K, B = q["M"], q["K"], q["B"]
    N = n_t - 1 if CN else n_t
    n_v, n_p = M.shape[0], sq["M_p"].shape[0]
    g = q["bc_values"]
    s = StokesSystem(M, K, B, sq["M_p"], sq["L_p"], n_t=n_t, beta=q["beta"], CN=CN, time_interval=q["time_interval"],
                     bc_dofs_v=bd)
    # host lifting, as incompressible_linear_solve does it
    l0, l1 = _host_lift(M, K, tau, n_t, CN, bd, g)
    lift = np.zeros((n_t, n_v))
    lift[:, bd] = g
    d10 = -tau * (B @ (lift[1:] if CN else lift).T).T
    if CN:
        d10 = kkt.apply_T_2(d10)
    rng = np.random.default_rng(SEED + 3)
    x0, x1 = rng.standard_normal((2 * N, n_v)), rng.standard_normal((2 * N, n_p))
    b = s.to_device(x0, x1)
    s.lift_bc_device(torch.from_numpy(g).to(s.device), b)
    c0, c1 = s.to_host_blocks(b)
    e0, e1 = np.concatenate([l0, l1]), np.concatenate([d10, np.zeros((N, n_p))])
    scale = max(np.abs(e0).max(), np.abs(e1).max())
    assert np.abs((c0 - x0) - e0).max() <= 1e-13 * scale and np.abs((c1 - x1) - e1).max() <= 1e-13 * scale
    assert np.array_equal(c0[:, bd], x0[:, bd])
    # solve from homogeneous host rows + the device lifting
    b_0_0, b_0_1 = kkt.build_rhs(M, K, tau, n_t, CN, bd, q["v_d"], q["f"], q["v_0"])
    b = s.to_device(np.concatenate([b_0_0, b_0_1]), np.zeros((2 * N, n_p)))
    s.lift_bc_device(g, b)
    s.setup_preconditioner(lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"])
    u = torch.zeros_like(b)
    info = s.solve_device(b, u)
    assert info.reason > 0 and info.its <= 40
    u0, _ = s.to_host_blocks(u)
    if CN:
        v = np.concatenate([q["v_0"][None], u0[:N]])
    else:
        v = u0[:N].copy()
    v[:, bd] = g
    err = kat.l2_error(M, v, q["true_v"]) / kat.l2_error(M, q["true_v"], 0 * q["true_v"])
    assert err < (1e-4 if CN else 1e-3)
    s.close()


@pytest.mark.gpu
def test_lift_bc_argument_and_state_errors():
    """NULL g with Dirichlet dofs, a call before ctl_assemble, an unknown layout: each returns its code and message,
    and the handle stays usable."""
    import torch
    from control_b200 import MultiBlockSystem
    from control_b200 import _lib as L
    lib = L.load()
    q = kat.heat_problem(6, 4, True, beta=1e-2)
    M, K, bd = q["M"], q["K"], q["bdofs"].astype(np.int32)
    s = MultiBlockSystem(M, K, n_t=4, beta=q["beta"], CN=True, time_interval=q["time_interval"], bc_dofs=bd)
    b = s.new_vector()
    assert lib.ctl_lift_bc(s._h, None, b.data_ptr(), L.CTL_LAYOUT_BLOCK_MAJOR) == -1
    assert b"null g" in lib.ctl_last_error(s._h)
    assert lib.ctl_lift_bc(s._h, b.data_ptr(), b.data_ptr(), 7) == -1
    assert b"layout" in lib.ctl_last_error(s._h)
    with pytest.raises(ValueError):
        s.lift_bc_device(np.zeros((3, bd.size)), b)
    g = np.ones((4, bd.size))
    s.lift_bc_device(g, b)                                   # still usable
    assert float(b.abs().sum()) > 0.0
    # values changed, not yet assembled
    data = sp.csr_matrix(M).sorted_indices().data.copy()
    assert lib.ctl_set_values(s._h, L.CTL_MAT_M, -1, data.ctypes.data) == 0
    g_dev = torch.ones(4 * bd.size, dtype=torch.float64, device=s.device)
    assert lib.ctl_lift_bc(s._h, g_dev.data_ptr(), b.data_ptr(), L.CTL_LAYOUT_BLOCK_MAJOR) == -3
    assert b"ctl_assemble" in lib.ctl_last_error(s._h)
    assert lib.ctl_assemble(s._h) == 0
    b2 = s.new_vector()
    s.lift_bc_device(g, b2)
    torch.cuda.synchronize()
    assert torch.equal(b, b2)
    # no Dirichlet dofs: nothing to do, g may be NULL
    s0 = MultiBlockSystem(M, K, n_t=4, beta=q["beta"], CN=True, time_interval=q["time_interval"])
    z = s0.new_vector()
    assert lib.ctl_lift_bc(s0._h, None, z.data_ptr(), L.CTL_LAYOUT_BLOCK_MAJOR) == 0
    assert float(z.abs().sum()) == 0.0
    s0.close()
    s.close()
