"""Multi-rank GPU check, launched by torchrun (one rank per GPU): the row-partitioned KKT
apply, preconditioner and solve must reproduce the single-rank oracle results."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import kat  # noqa: E402
from control_b200 import MultiBlockSystem, partition  # noqa: E402
from oracle import control as ocontrol  # noqa: E402
from oracle import kkt  # noqa: E402
from oracle import pc as opc  # noqa: E402


def rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    # a small dense coarsest level, so that the hierarchy has several levels at this size; MP_NX / CTL_AMG_REP_NNZ
    # choose how many of them are distributed (halo.cu)
    amg = dict(coarse_max=int(os.environ.get("MP_COARSE_MAX", "30")))
    nx = int(os.environ.get("MP_NX", "40"))
    for CN in (True, False):
        q = kat.heat_problem(nx, 9, CN, beta=1e-3)
        n = q["M"].shape[0]
        s = MultiBlockSystem(q["M"], q["K"], n_t=q["n_t"], beta=q["beta"], CN=CN,
                             time_interval=q["time_interval"], bc_dofs=q["bdofs"], rank=rank, world=world)
        s.init_comm(dist)
        assert (s.row_begin, s.n_local) == partition.ownership_range(n, world, rank)
        rng = np.random.default_rng(0)
        x0 = rng.standard_normal((s.N, n))
        x1 = rng.standard_normal((s.N, n))
        y0, y1 = kkt.kkt_apply_fused(q["M"], q["K"], s.tau, q["beta"], q["n_t"], CN, q["bdofs"], x0, x1)
        loc = lambda a: partition.local_blocks(a, n, world, rank)
        g0, g1 = s.to_host_blocks(s.apply(s.to_device(loc(x0), loc(x1))))
        e_apply = max(rel(g0, loc(y0)), rel(g1, loc(y1)))
        assert e_apply < 1e-13, e_apply
        # preconditioner
        s.setup_preconditioner(lambda_v_bounds=q["lambda_v_bounds"], **amg)
        pc = opc.construct_pc(q["M"], q["K"], q["tau"], q["beta"], q["n_t"], CN, q["bdofs"],
                              lambda_v_bounds=q["lambda_v_bounds"], amg_params=amg)
        b0, b1 = x0.copy(), x1.copy()
        b0[:, q["bdofs"]] = 0.0
        b1[:, q["bdofs"]] = 0.0
        r0, r1 = pc(b0, b1)
        p0, p1 = s.to_host_blocks(s.pc_apply(s.to_device(loc(b0), loc(b1)), raw=True))
        e_pc = max(rel(p0, loc(r0)), rel(p1, loc(r1)))
        assert e_pc < 1e-10, e_pc
        # solve
        # BE stalls near 1e-8 (rounding floor, see test_gpu_pc.py): compare counts above it
        sp_ = {"linear_solver": "fgmres", "maximum_iterations": 100, "relative_tolerance": 1e-8 if CN else 1e-6,
               "absolute_tolerance": 0.0, "gmres_restart": 100}
        ref = ocontrol.linear_solve(q["M"], q["K"], beta=q["beta"], n_t=q["n_t"], CN=CN,
                                    time_interval=q["time_interval"], bdofs=q["bdofs"], v_d=q["v_d"],
                                    f=q["f"], lambda_v_bounds=q["lambda_v_bounds"], solver_parameters=sp_, amg_params=amg)
        u0 = np.zeros((s.N, s.n_local))
        u1 = np.zeros((s.N, s.n_local))
        info = s.solve(u0, u1, loc(ref["b_0"]), loc(ref["b_1"]), solver_parameters=sp_, pc_fn="builtin")
        e_sol = max(rel(u0, loc(ref["v_blocks"])), rel(u1, loc(ref["zeta_blocks"])))
        assert info.reason > 0 and abs(info.its - ref["ksp"].its) <= 1, (info.its, ref["ksp"].its)
        assert e_sol < (1e-6 if CN else 1e-4), e_sol
        # right-hand sides from nodal data and the objective on this rank's rows (ctl_build_rhs, ctl_objective)
        n_t = q["n_t"]
        f_nodal = rng.standard_normal((n_t, n))
        v_hat = q["v_hat"] + 0.1 * rng.standard_normal(q["v_hat"].shape)
        v_0 = rng.standard_normal(n)
        v_0[q["bdofs"]] = 0.0
        rows = slice(s.row_begin, s.row_begin + s.n_local)
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a[:, rows])).to(s.device)
        bd_ = s.build_rhs_device(dev(v_hat), dev(f_nodal), v_0)
        d0, d1 = s.to_host_blocks(bd_)
        r0, r1 = kkt.build_rhs(q["M"], q["K"], q["tau"], n_t, CN, q["bdofs"], (q["M"] @ v_hat.T).T, (q["M"] @ f_nodal.T).T, v_0)
        e_rhs = max(np.abs(d0 - loc(r0)).max(), np.abs(d1 - loc(r1)).max()) / max(np.abs(r0).max(), np.abs(r1).max())
        assert e_rhs < 1e-13, e_rhs
        vv, zz = rng.standard_normal((n_t, n)), rng.standard_normal((n_t, n))
        J_dev = s.objective_device(dev(vv), dev(zz), dev(v_hat))
        J_ref = ocontrol.objective(q["M"], vv, zz, v_hat, q["tau"], q["beta"], CN)
        assert abs(J_dev - J_ref) <= 1e-12 * abs(J_ref), (J_dev, J_ref)
        if rank == 0:
            print(f"CN={CN} world={world} nx={nx} rhs {e_rhs:.1e} J {abs(J_dev - J_ref) / abs(J_ref):.1e}", flush=True)
        if rank == 0:
            print(f"CN={CN} world={world} nx={nx} levels {s._lib.ctl_amg_num_levels(s._h, 0)}: apply {e_apply:.1e} pc {e_pc:.1e} solve its {info.its}/{ref['ksp'].its} "
                  f"diff {e_sol:.1e}", flush=True)
        s.close()
    dist.barrier()
    if rank == 0:
        print("MP_GPU_CHECK_OK", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
