"""Full heat-control KKT solve at a chosen size (default: BASELINE config C2)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=1024)
    ap.add_argument("--n_t", type=int, default=64)
    ap.add_argument("--ksp", default="fgmres")
    ap.add_argument("--mode", default="triangular")
    ap.add_argument("--rtol", type=float, default=1e-6)
    ap.add_argument("--restart", type=int, default=30)
    ap.add_argument("--be", action="store_true")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--dim", type=int, default=2)
    ap.add_argument("--amg", default="", help="comma list key=value of AMG options (cycles, nu, lo, hi, acc_lo, ...)")
    args = ap.parse_args()
    from synthetic import problems as kat
    from control_b200 import MultiBlockSystem
    from control_b200.control import build_rhs
    t = time.time()
    q = kat.heat_problem(args.nx, args.n_t, not args.be) if args.dim == 2 else kat.heat_problem_3d(args.nx, args.n_t, not args.be)
    print(f"assembled n={q['M'].shape[0]} in {time.time() - t:.1f}s", flush=True)
    t = time.time()
    s = MultiBlockSystem(q["M"], q["K"], n_t=q["n_t"], beta=q["beta"], CN=not args.be,
                         time_interval=q["time_interval"], bc_dofs=q["bdofs"])
    print(f"system created in {time.time() - t:.1f}s", flush=True)
    t = time.time()
    amg = {}
    for kv in filter(None, args.amg.split(",")):
        k, v = kv.split("=")
        amg[k] = float(v) if "." in v else int(v)
    s.setup_preconditioner(lambda_v_bounds=q["lambda_v_bounds"], mode=args.mode, **amg)
    print(f"pc setup in {time.time() - t:.1f}s; levels:",
          [s._lib.ctl_amg_num_levels(s._h, i) for i in range(s._lib.ctl_amg_num_hierarchies(s._h))], flush=True)
    b0, b1 = build_rhs(q["M"], q["K"], q["tau"], q["n_t"], not args.be, q["bdofs"], q["v_d"], q["f"],
                           np.zeros(s.n))
    b = s.to_device(b0, b1)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                          str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    print(f"gpu: {gpu}", flush=True)
    sp_ = {"linear_solver": args.ksp, "gmres_restart": args.restart, "maximum_iterations": 60, "preconditioner": True,
           "relative_tolerance": args.rtol, "absolute_tolerance": 0.0}
    for rep in range(args.reps):
        u = s.new_vector()
        l0 = s.kernel_launches()
        info = s.solve_device(b, u, solver_parameters=sp_, pc="builtin")
        print(json.dumps({"its": info.its, "reason": info.reason, "seconds": info.seconds_total,
                          "mult_s": info.seconds_mult, "pc_s": info.seconds_pc,
                          "vector_s": info.seconds_total - info.seconds_mult - info.seconds_pc, "n_mult": info.n_mult,
                          "n_pc": info.n_pc, "launches": s.kernel_launches() - l0,
                          "res": s.residual_norm(b, u), "hist": info.history[:3] + info.history[-2:]}), flush=True)
    print("mem GB", torch.cuda.max_memory_allocated() / 1e9, torch.cuda.mem_get_info())


if __name__ == "__main__":
    main()
