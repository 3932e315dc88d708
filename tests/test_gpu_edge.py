"""Edge cases of the solve path on the GPU against the oracle: single time block, no
constrained dofs, zero right-hand side, warm start, short restart, error reporting."""
import numpy as np
import pytest

import kat
from oracle import control as ocontrol
from oracle import kkt
from synthetic import fem

pytestmark = pytest.mark.gpu


def _solve_both(q, CN, sp_, **kw):
    from control_b200 import MultiBlockSystem
    ref = ocontrol.linear_solve(q["M"], q["K"], beta=q["beta"], n_t=q["n_t"], CN=CN,
                                time_interval=q["time_interval"], bdofs=q["bdofs"], v_d=q["v_d"], f=q["f"],
                                lambda_v_bounds=q["lambda_v_bounds"], solver_parameters=sp_, **kw)
    s = MultiBlockSystem(q["M"], q["K"], n_t=q["n_t"], beta=q["beta"], CN=CN,
                         time_interval=q["time_interval"], bc_dofs=q["bdofs"])
    s.setup_preconditioner(lambda_v_bounds=q["lambda_v_bounds"])
    u0 = np.zeros((s.N, s.n))
    u1 = np.zeros((s.N, s.n))
    info = s.solve(u0, u1, ref["b_0"], ref["b_1"], solver_parameters=sp_, pc_fn="builtin")
    return s, info, u0, u1, ref


@pytest.mark.parametrize("CN", [True, False])
def test_two_time_levels(CN):
    """n_t = 2: a single block for CN (no T coupling at all), two for BE."""
    q = kat.heat_problem(9, 2, CN, beta=1e-2)
    sp_ = {"linear_solver": "fgmres", "maximum_iterations": 100, "relative_tolerance": 1e-7,
           "absolute_tolerance": 0.0, "gmres_restart": 100}
    s, info, u0, u1, ref = _solve_both(q, CN, sp_)
    assert s.N == (1 if CN else 2)
    assert info.reason > 0 and abs(info.its - ref["ksp"].its) <= 1
    assert np.abs(u0 - ref["v_blocks"]).max() < 1e-5 * np.abs(ref["v_blocks"]).max()
    s.close()



@pytest.mark.parametrize("CN", [True, False])
def test_kkt_apply_with_rows_too_long_to_stage(CN):
    """One extra dof coupled to every dof of a 12 x 12 P1 mesh (a symmetric dense row and column of M and K): its row
    has 170 entries, more than the 128 per row that the staged KKT kernel can hold (kkt_apply.cu: STAGE_CAP entries
    for at least 8 rows per CTA), so the apply runs the unstaged kernel."""
    import scipy.sparse as sp
    from control_b200 import MultiBlockSystem
    q = kat.heat_problem(12, 6, CN)
    n0 = q["M"].shape[0]
    assert n0 + 1 > 128
    rng = np.random.default_rng(5)

    def bordered(A, scale):
        c = sp.csr_matrix(scale * rng.uniform(0.5, 1.0, (n0, 1)))
        B = sp.bmat([[sp.csr_matrix(A), c], [c.T, sp.csr_matrix([[scale * n0]])]], format="csr")
        B.sort_indices()
        return B

    M, K, bd = bordered(q["M"], 1e-3), bordered(q["K"], 1e-1), q["bdofs"]
    s = MultiBlockSystem(M, K, n_t=q["n_t"], beta=q["beta"], CN=CN, time_interval=q["time_interval"], bc_dofs=bd)
    assert s.N <= 64                                       # the narrow kernels (one block of ld <= 64 columns)
    x0 = rng.standard_normal((s.N, s.n))
    x1 = rng.standard_normal((s.N, s.n))
    y0, y1 = kkt.kkt_apply_fused(M, K, s.tau, q["beta"], q["n_t"], CN, bd, x0, x1)
    g0, g1 = s.to_host_blocks(s.apply(s.to_device(x0, x1)))
    err = max(np.abs(g0 - y0).max(), np.abs(g1 - y1).max()) / max(np.abs(y0).max(), np.abs(y1).max())
    assert err < 1e-13, err
    s.close()

def test_no_constrained_dofs():
    q = kat.heat_problem(8, 5, True, beta=1e-2)
    q["bdofs"] = np.zeros(0, dtype=np.int32)
    sp_ = {"linear_solver": "fgmres", "maximum_iterations": 100, "relative_tolerance": 1e-8, "absolute_tolerance": 0.0}
    s, info, u0, u1, ref = _solve_both(q, True, sp_)
    assert info.reason > 0 and abs(info.its - ref["ksp"].its) <= 1
    assert np.abs(u1 - ref["zeta_blocks"]).max() < 1e-6 * np.abs(ref["zeta_blocks"]).max()
    s.close()


def test_zero_rhs_warm_start_and_short_restart():
    q = kat.heat_problem(10, 6, True, beta=1e-3)
    sp_ = {"linear_solver": "gmres", "gmres_restart": 3, "maximum_iterations": 100,
           "relative_tolerance": 1e-8, "absolute_tolerance": 0.0}
    s, info, u0, u1, ref = _solve_both(q, True, sp_)
    # GMRES(3): many restarts, left preconditioning, preconditioned norm
    assert info.reason > 0 and abs(info.its - ref["ksp"].its) <= 1
    k = min(len(info.history), len(ref["ksp"].history)) - 1
    assert np.allclose(info.history[:k], ref["ksp"].history[:k], rtol=1e-6)
    # warm start from the solution: the initial residual already passes the test (0 iterations)
    info2 = s.solve(u0, u1, ref["b_0"], ref["b_1"], solver_parameters=dict(sp_, relative_tolerance=1e-6), pc_fn="builtin")
    assert info2.its == 0 and info2.reason > 0
    # zero right-hand side, zero guess: PETSc's default test converges at iteration 0
    z0 = np.zeros_like(u0)
    z1 = np.zeros_like(u1)
    info3 = s.solve(z0, z1, np.zeros_like(u0), np.zeros_like(u1), solver_parameters=sp_, pc_fn="builtin")
    assert info3.its == 0 and info3.reason > 0 and not z0.any() and not z1.any()
    s.close()


def test_state_errors_are_loud():
    from control_b200 import CtlError, MultiBlockSystem
    q = kat.heat_problem(5, 4, True)
    s = MultiBlockSystem(q["M"], q["K"], n_t=q["n_t"], beta=q["beta"], CN=True,
                         time_interval=q["time_interval"], bc_dofs=q["bdofs"])
    sp_ = {"linear_solver": "fgmres", "relative_tolerance": 1e-6, "absolute_tolerance": 0.0}
    b = np.zeros((s.N, s.n))
    with pytest.raises(CtlError):                      # in-built PC requested before setup
        s.solve(b.copy(), b.copy(), b, b, solver_parameters=sp_, pc_fn="builtin")
    with pytest.raises(ValueError):                    # wrong vector size
        s.to_device(np.zeros(7))
    with pytest.raises(ValueError):                    # unsupported Krylov type
        s.solve(b.copy(), b.copy(), b, b, solver_parameters=dict(sp_, linear_solver="cg"))
    with pytest.raises(KeyError):                      # required keys, preconditioner.py:739-740
        s.solve(b.copy(), b.copy(), b, b, solver_parameters={"linear_solver": "fgmres"})
    with pytest.raises(CtlError):                      # diagonal mode needs CN + symmetric K
        K2 = q["K"].copy()
        K2.data = K2.data * (1.0 + 0.1 * np.random.default_rng(0).standard_normal(K2.nnz))
        s2 = MultiBlockSystem(q["M"], K2, n_t=q["n_t"], beta=q["beta"], CN=True, bc_dofs=q["bdofs"])
        s2.setup_preconditioner(mode="diagonal")
    s.close()


def test_solve_host_entry_point_matches_device_solve():
    """ctl_solve_host (host buffers in, host buffers out) == ctl_solve on device vectors."""
    from control_b200 import MultiBlockSystem
    q = kat.heat_problem(12, 7, True, beta=1e-3)
    sp_ = {"linear_solver": "fgmres", "maximum_iterations": 100, "relative_tolerance": 1e-9, "absolute_tolerance": 0.0}
    s, info, u0, u1, ref = _solve_both(q, True, sp_)
    b = np.concatenate([ref["b_0"].ravel(), ref["b_1"].ravel()])
    u = np.zeros_like(b)
    info_h = s.solve_host(u, b, solver_parameters=sp_)
    assert info_h.its == info.its and info_h.reason == info.reason
    assert np.array_equal(u, np.concatenate([u0.ravel(), u1.ravel()]))      # same kernels, same order: bit-identical
    with pytest.raises(ValueError):
        s.solve_host(u[:-1], b, solver_parameters=sp_)
    s.close()
