"""Multi-rank GPU check of the Stokes control path, launched by torchrun (one rank per GPU): the row-partitioned
outer operator, in-built preconditioner, solve, lifting and Picard residual against the single-rank oracle, and the
Stokes drivers of ``Control.Instationary`` on several ranks against the same drivers on one rank.  Every check is
printed by rank 0; the run ends with MP_STOKES_CHECK_OK when all of them hold."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kat  # noqa: E402
import test_nonlinear_device_loops as nl  # noqa: E402
from control_b200 import Control, partition  # noqa: E402
from control_b200.stokes import StokesSystem  # noqa: E402
from oracle import stokes as ostokes  # noqa: E402
from synthetic import fem, problems  # noqa: E402

LAMBDA_V = (0.3924, 2.0598)      # as tests/test_gpu_stokes.py
LAMBDA_P = (0.5, 2.0)
AMG = dict(coarse_max=40)
AMG_P = dict(coarse_max=20)

failures = []


def rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def check(rank, name, value, ok):
    if rank == 0:
        print(f"{name}: {value}  {'ok' if ok else 'FAILED'}", flush=True)
    if not ok:
        failures.append(name)


def same_on_all_ranks(x):
    parts = [None] * dist.get_world_size()
    dist.all_gather_object(parts, x)
    return all(p == parts[0] for p in parts)


def operator_pc_solve(rank, world, CN, nx, n_t):
    th = fem.assemble_taylor_hood_2d(nx, nx, 1.0, 1.0)
    beta, tau, N = 1e-2, 1.0 / (n_t - 1.0), n_t - 1 if CN else n_t
    bd = th["bdofs_v"]
    s = StokesSystem(th["M_v"], th["K_v"], th["B"], th["M_p"], th["K_p"], n_t=n_t, beta=beta, CN=CN, bc_dofs_v=bd,
                     rank=rank, world=world)
    s.init_comm(dist)
    n_v, n_p = s.n_v, s.n_p
    assert (s.velocity_rows.start, s.n_v_local) == partition.ownership_range(n_v, world, rank)
    assert (s.pressure_rows.start, s.n_p_local) == partition.ownership_range(n_p, world, rank)
    lv = lambda a: np.ascontiguousarray(a[:, s.velocity_rows])
    lp = lambda a: np.ascontiguousarray(a[:, s.pressure_rows])
    tag = f"CN={CN} world={world} nx={nx} n_t={n_t}"
    rng = np.random.default_rng(11)
    # operator
    x0, x1 = rng.standard_normal((2 * N, n_v)), rng.standard_normal((2 * N, n_p))
    y0, y1 = s.to_host_blocks(s.apply(s.to_device(lv(x0), lp(x1))))
    r0, r1 = ostokes.stokes_apply_fused(th["M_v"], th["K_v"], th["B"], tau, beta, n_t, CN, bd, x0, x1)
    e = max(rel(y0, lv(r0)), rel(y1, lp(r1)))
    check(rank, f"{tag} apply vs stokes_apply_fused", f"{e:.1e}", e < 1e-13)
    # preconditioner
    s.setup_preconditioner(lambda_v_bounds=LAMBDA_V, lambda_p_bounds=LAMBDA_P, amg=AMG, amg_p=AMG_P)
    pc = ostokes.construct_stokes_pc(th["M_v"], th["K_v"], th["B"], th["M_p"], th["K_p"], tau, beta, n_t, CN, bd,
                                     lambda_v_bounds=LAMBDA_V, lambda_p_bounds=LAMBDA_P, inner="amg", amg_params=AMG,
                                     amg_params_p=AMG_P)
    b0 = rng.standard_normal((2 * N, n_v))
    b0[:, bd] = 0.0
    b1 = rng.standard_normal((2 * N, n_p))
    b1 -= b1.mean(axis=1, keepdims=True)
    u0, u1 = s.to_host_blocks(s.pc_apply(s.to_device(lv(b0), lp(b1)), raw=True))
    o0, o1 = pc(b0, b1)
    e = max(rel(u0, lv(o0)), rel(u1, lp(o1)))
    check(rank, f"{tag} pc_fn vs construct_stokes_pc", f"{e:.1e}", e < 1e-10)
    # solve
    xr0 = rng.standard_normal((2 * N, n_v))
    xr0[:, bd] = 0.0
    xr1 = rng.standard_normal((2 * N, n_p))
    xr1 -= xr1.mean(axis=1, keepdims=True)
    c0, c1 = ostokes.stokes_apply_fused(th["M_v"], th["K_v"], th["B"], tau, beta, n_t, CN, bd, xr0, xr1)
    sp_ = {"linear_solver": "fgmres", "maximum_iterations": 300, "relative_tolerance": 1e-8 if CN else 1e-6,
           "absolute_tolerance": 0.0, "gmres_restart": 100, "monitor_convergence": False}
    w0, w1 = np.zeros((2 * N, s.n_v_local)), np.zeros((2 * N, s.n_p_local))
    info = s.solve(w0, w1, lv(c0), lp(c1), solver_parameters=sp_)
    g0, g1, res = ostokes.stokes_solve(th["M_v"], th["K_v"], th["B"], th["M_p"], th["K_p"], beta=beta, n_t=n_t, CN=CN,
                                       bdofs_v=bd, b_0=c0, b_1=c1, solver_parameters=sp_, pc_fn=pc)
    check(rank, f"{tag} solve its vs stokes_solve", f"{info.its} / {res.its}",
          info.reason > 0 and abs(info.its - res.its) <= 1)
    e = rel(np.concatenate([w0.ravel(), w1.ravel()]), np.concatenate([lv(g0).ravel(), lp(g1).ravel()]))
    check(rank, f"{tag} solve solution vs stokes_solve", f"{e:.1e}", e < (1e-6 if CN else 1e-4))
    launches = s.kernel_launches()
    s.close()
    return launches


def lift_and_residual(rank, world, CN):
    c = nl._ns_case(CN)
    q, N, bd = c["q"], c["N"], c["q"]["bdofs"]
    s = StokesSystem(q["M"], q["D_v"](np.zeros(c["n_v"]), 0.0), q["B"], q["sq"]["M_p"], q["sq"]["L_p"], n_t=q["n_t"],
                     beta=q["beta"], CN=CN, time_interval=q["time_interval"], bc_dofs_v=bd,
                     D_p=q["D_p"](np.zeros(c["n_v"]), 0.0), rank=rank, world=world)
    s.init_comm(dist)
    lv = lambda a: np.ascontiguousarray(a[:, s.velocity_rows])
    lp = lambda a: np.ascontiguousarray(a[:, s.pressure_rows])
    tag = f"CN={CN} world={world} Navier-Stokes iterate"
    s.set_forward(c["K_it"], c["P_it"])
    b = s.lift_bc_device(c["g"], s.to_device(lv(c["b_hom"][0]), lp(c["b_hom"][1])))
    h0, h1 = nl._host_lifted_b(c)
    d0, d1 = s.to_host_blocks(b)
    scale = max(np.abs(h0).max(), np.abs(h1).max())
    e = max(np.abs(d0 - lv(h0)).max(), np.abs(d1 - lp(h1)).max()) / scale
    check(rank, f"{tag} lift_bc vs host lifting", f"{e:.1e}", e <= 1e-12)
    x = s.to_device(lv(c["x0"]), lp(c["x1"]))
    r = s.new_vector()
    norm = s.nonlinear_residual(b, x, r)
    r0, r1 = s.to_host_blocks(r)
    scale = max(np.abs(c["e0"]).max(), np.abs(c["e1"]).max())
    e = max(np.abs(r0 - lv(c["e0"])).max(), np.abs(r1 - lp(c["e1"])).max()) / scale
    check(rank, f"{tag} nonlinear_residual vs res_eval", f"{e:.1e}", e <= 1e-12)
    e = abs(norm - c["ref_norm"]) / c["ref_norm"]
    check(rank, f"{tag} residual norm vs res_eval", f"{e:.1e}", e <= 1e-12)
    check(rank, f"{tag} residual norm bitwise equal on every rank", repr(norm), same_on_all_ranks(norm))
    s.close()


def linear_driver(rank, world, CN, nx, n_t):
    q = problems.stokes_problem(nx, n_t, CN, beta=1e-2)
    th = q["th"]

    def level(t):
        return int(round(t / q["tau"]))
    out = []
    sp_ = {"linear_solver": "fgmres", "maximum_iterations": 300, "relative_tolerance": 1e-10 if CN else 1e-8,
           "absolute_tolerance": 0.0, "gmres_restart": 100, "monitor_convergence": False}
    for w, r in ((1, 0), (world, rank)):
        c = Control.Instationary(q["M"], q["K"], desired_state=lambda t: (q["v_d"][level(t)], q["v_hat"][level(t)]),
                                 force_f=lambda t: q["f"][level(t)], beta=q["beta"], CN=CN, n_t=n_t,
                                 time_interval=q["time_interval"], bc_dofs=q["bdofs"], rank=r, world=w)
        ksp = c.incompressible_linear_solve("constant", space_p=dict(B=th["B"], M_p=th["M_p"], K_p=th["K_p"]),
                                            solver_parameters=dict(sp_), lambda_v_bounds=q["lambda_v_bounds"],
                                            lambda_p_bounds=q["lambda_p_bounds"], amg=AMG, amg_p=AMG_P,
                                            print_error=False)
        out.append((ksp.its, np.concatenate([c._v.ravel(), c._zeta.ravel()]), np.concatenate([c._p.ravel(), c._mu.ravel()])))
        c.close()
    (i1, v1, p1), (iw, vw, pw) = out
    tag = f"CN={CN} incompressible_linear_solve world={world} vs 1 (nx={nx})"
    check(rank, f"{tag} its", f"{iw} / {i1}", iw == i1)
    e = max(rel(vw, v1), rel(pw, p1))
    check(rank, f"{tag} solution", f"{e:.1e}", e < 1e-8)


def picard(rank, world, CN):
    # 6 x 6 Q2-Q1 cells (n_v = 338, n_p = 49) with the small coarse sizes of the other steps: a hierarchy on several
    # ranks needs at least two levels (amg_build), which the default coarse_max of 2500 would not give
    q = kat.reference_navier_stokes_problem(CN, nx=6, n_t=6)

    def level(t):
        return int(round(t / q["tau"]))
    space_p = dict(B=q["B"], M_p=q["sq"]["M_p"], K_p=q["sq"]["L_p"],
                   forward_matrix_p=lambda v_i, t, gauss_newton: q["D_p"](v_i, t))
    out = []
    for w, r in ((1, 0), (world, rank)):
        c = Control.Instationary(q["M"], lambda v_i, t, gauss_newton: q["D_v"](v_i, t),
                                 desired_state=lambda t: (q["v_d"][level(t)], q["v_hat"][level(t)]), beta=q["beta"],
                                 n_t=q["n_t"], CN=CN, time_interval=q["time_interval"], bc_dofs=q["bdofs"],
                                 bc_values=lambda t: q["bc_values"][level(t)], rank=r, world=w)
        c.incompressible_non_linear_solve("constant", space_p=space_p, solver_parameters=dict(nl._NS_SP),
                                          amg=AMG, amg_p=AMG_P, max_non_linear_iter=3, relative_non_linear_tol=1e-14,
                                          absolute_non_linear_tol=0.0, print_error_non_linear=False, device_loop=False)
        out.append((list(c.inner_iterations), np.array(c.non_linear_history)))
        c.close()
    (i1, h1), (iw, hw) = out
    tag = f"CN={CN} Navier-Stokes host Picard loop world={world} vs 1"
    check(rank, f"{tag} inner its", f"{iw} / {i1}", iw == i1 and len(i1) == 3)
    e = rel(hw, h1) if hw.shape == h1.shape else np.inf
    check(rank, f"{tag} history", f"{e:.1e} {list(hw)}", e < 1e-6)


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = int(os.environ["LOCAL_RANK"])          # one GPU per rank: NCCL refuses two ranks on one device
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
    nx, n_t = int(os.environ.get("MP_NX", "8")), int(os.environ.get("MP_NT", "5"))
    if rank == 0:
        print(f"{torch.cuda.get_device_name()} x {world}", flush=True)
    for CN in (True, False):
        for step in (lambda: operator_pc_solve(rank, world, CN, nx, n_t), lambda: lift_and_residual(rank, world, CN),
                     lambda: linear_driver(rank, world, CN, nx, n_t), lambda: picard(rank, world, CN)):
            try:
                step()
            except Exception as e:       # report and go on: one run shows every check
                import traceback
                traceback.print_exc()
                failures.append(f"rank {rank}: {type(e).__name__}: {e}")
            dist.barrier()
    failed = [None] * world
    dist.all_gather_object(failed, failures)
    if rank == 0:
        bad = [f for part in failed for f in part]
        print("FAILURES: " + "; ".join(bad) if bad else "MP_STOKES_CHECK_OK", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
