"""Block-scalar velocity sweeps against the vector path at BASELINE config C4 (Taylor-Hood P2-P1 512 x 512, n_t = 32,
CN, FGMRES + pressure-Schur preconditioner), in ONE process: the problem is built once, then the arms alternate velocity
block size 1, 2, 1, 2.  Each arm creates the StokesSystem, sets up the preconditioner, times a cold velocity inner solve
and the level-0 smoother step (ctl_time_amg, operands larger than L2), runs one full solve and closes the system.

Prints one JSON line per arm and a last line with the card's name and power limit, read in the same call:
  setup_s           ctl_stokes_pc_setup wall time (host AMG set-up included)
  pc_block_size     block size the velocity sweeps actually ran with
  smoother_ms/_MB   level-0 Chebyshev step: time and algorithmic bytes (matrix once, vectors bs times)
  inner_ms/_MB      one velocity inner solve (all cycles, all levels): time and algorithmic bytes
  level0_matrix_MB  matrix stream of one level-0 product; level0_B_per_entry tells the SELL format chosen for it
                    (plain f64 12, 16-bit offsets 10, dictionary codes 1-2, stencil slices about 0.1)
  its, solve_s, true_res, rel_res   the outer solve"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=512)
    ap.add_argument("--n_t", type=int, default=32)
    ap.add_argument("--arms", default="1,2,1,2", help="velocity block size of each arm, in order")
    ap.add_argument("--reps", type=int, default=20, help="launches per ctl_time_amg measurement")
    ap.add_argument("--rtol", type=float, default=1e-6)
    ap.add_argument("--restart", type=int, default=30)
    ap.add_argument("--max_it", type=int, default=100)
    args = ap.parse_args()
    from control_b200.control import build_rhs
    from control_b200.stokes import StokesSystem
    from synthetic import problems
    t = time.time()
    q = problems.stokes_problem(args.nx, args.n_t, True)
    th = q["th"]
    b00, b01 = build_rhs(q["M"], q["K"], q["tau"], q["n_t"], True, q["bdofs"], q["v_d"], q["f"], np.zeros(th["M_v"].shape[0]))
    print(json.dumps({"assembled_s": round(time.time() - t, 1), "n_v": th["M_v"].shape[0], "n_p": th["M_p"].shape[0]}),
          flush=True)
    sp_ = {"linear_solver": "fgmres", "gmres_restart": args.restart, "maximum_iterations": args.max_it,
           "preconditioner": True, "relative_tolerance": args.rtol, "absolute_tolerance": 0.0}
    for bs in [int(a) for a in args.arms.split(",")]:
        s = StokesSystem(th["M_v"], th["K_v"], th["B"], th["M_p"], th["K_p"], n_t=q["n_t"], beta=q["beta"], CN=True,
                         time_interval=q["time_interval"], bc_dofs_v=q["bdofs"], velocity_block_size=bs)
        torch.cuda.synchronize()
        t = time.time()
        s.setup_preconditioner(lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"])
        torch.cuda.synchronize()
        setup_s = time.time() - t
        v, lib = s.velocity, s._lib
        out = (C.c_double * 7)()
        v._call(lib.ctl_time_amg, 0, args.reps, 1, out)
        n0, nnz0, nnzp = C.c_int32(), C.c_int64(), C.c_int64()
        v._check(lib.ctl_amg_level_size(v._h, 0, 0, C.byref(n0), C.byref(nnz0), C.byref(nnzp)))
        nc = v.pc_block_size
        mat0 = out[1] - (8.0 + 32.0 * nc) * n0.value
        b = s.to_device(np.concatenate([b00, b01]), np.zeros((2 * s.N, s.n_p)))
        u = torch.zeros_like(b)
        torch.cuda.synchronize()
        t = time.time()
        info = s.solve_device(b, u, solver_parameters=sp_)
        torch.cuda.synchronize()
        solve_s = time.time() - t
        r = b - s.apply(u)
        r0, r1 = s.to_host_blocks(r)
        r0[:, q["bdofs"]] = 0.0
        r1 = r1 - r1.mean(axis=1, keepdims=True)
        res = float(np.sqrt((r0 ** 2).sum() + (r1 ** 2).sum()))
        bnorm = float(torch.linalg.vector_norm(b))
        print(json.dumps({"block_size": bs, "pc_block_size": nc, "setup_s": round(setup_s, 2),
                          "level0_rows": n0.value, "level0_entries": nnz0.value,
                          "levels": int(lib.ctl_amg_num_levels(v._h, 0)),
                          "smoother_ms": round(out[0], 4), "smoother_MB": round(out[1] / 1e6, 1),
                          "inner_ms": round(out[4], 4), "inner_MB": round(out[5] / 1e6, 1),
                          "inner_launches": int(out[6]), "level0_matrix_MB": round(mat0 / 1e6, 1),
                          "level0_B_per_entry": round(mat0 / max(nnz0.value, 1), 3),
                          "its": info.its, "reason": info.reason, "solve_s": round(solve_s, 2),
                          "pc_s": round(info.seconds_pc, 2), "n_pc": info.n_pc, "true_res": res,
                          "rel_res": res / bnorm}), flush=True)
        s.close()
        del s, b, u, r
        torch.cuda.empty_cache()
    power = None
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:      # the card's name from torch is still printed
        power = f"unavailable: {e}"
    print(json.dumps({"gpu": torch.cuda.get_device_name(), "name_power_limit": power}), flush=True)


if __name__ == "__main__":
    main()
