"""Instationary Stokes control solve at a chosen size (default: BASELINE config C4:
Taylor-Hood P2-P1 on 512x512, n_t = 32, CN, FGMRES + pressure-Schur preconditioner)."""
import argparse
import json
import os
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
    ap.add_argument("--beta", type=float, default=1.0)
    ap.add_argument("--rtol", type=float, default=1e-6)
    ap.add_argument("--restart", type=int, default=30)
    ap.add_argument("--be", action="store_true")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--max_it", type=int, default=100)
    ap.add_argument("--inner_its", type=int, default=5)
    ap.add_argument("--amg", default="", help="comma list key=value: velocity AMG options")
    ap.add_argument("--amg_p", default="", help="comma list key=value: K_p AMG options")
    ap.add_argument("--block-size", type=int, default=1,
                    help="velocity block size: 2 runs the velocity sweeps on the scalar block of I_2 (x) S")
    args = ap.parse_args()
    from synthetic import problems
    from control_b200.control import build_rhs
    from control_b200.stokes import StokesSystem
    t = time.time()
    q = problems.stokes_problem(args.nx, args.n_t, not args.be, beta=args.beta)
    th = q["th"]
    print(f"assembled n_v={th['M_v'].shape[0]} n_p={th['M_p'].shape[0]} nnz_v={th['M_v'].nnz} in {time.time() - t:.1f}s",
          flush=True)
    t = time.time()
    s = StokesSystem(th["M_v"], th["K_v"], th["B"], th["M_p"], th["K_p"], n_t=q["n_t"], beta=q["beta"], CN=not args.be,
                     time_interval=q["time_interval"], bc_dofs_v=q["bdofs"], velocity_block_size=args.block_size)
    print(f"system created in {time.time() - t:.1f}s", flush=True)
    t = time.time()
    def parse(txt):
        out = {}
        for kv in filter(None, txt.split(",")):
            k, v = kv.split("=")
            out[k] = float(v) if "." in v else int(v)
        return out
    s.setup_preconditioner(lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"],
                           inner_its=args.inner_its, amg=parse(args.amg), amg_p=parse(args.amg_p))
    print(f"pc setup in {time.time() - t:.1f}s, velocity sweeps with block size {s.velocity.pc_block_size}", flush=True)
    N = s.N
    b00, b01 = build_rhs(q["M"], q["K"], q["tau"], q["n_t"], not args.be, q["bdofs"], q["v_d"], q["f"], np.zeros(s.n_v))
    b = s.to_device(np.concatenate([b00, b01]), np.zeros((2 * N, s.n_p)))
    sp_ = {"linear_solver": "fgmres", "gmres_restart": args.restart, "maximum_iterations": args.max_it, "preconditioner": True,
           "relative_tolerance": args.rtol, "absolute_tolerance": 0.0}
    for rep in range(args.reps):
        u = torch.zeros_like(b)
        l0 = s.kernel_launches()
        info = s.solve_device(b, u, solver_parameters=sp_)
        r = b - s.apply(u)
        r0, r1 = s.to_host_blocks(r)
        r0[:, q["bdofs"]] = 0.0
        r1 = r1 - r1.mean(axis=1, keepdims=True)
        print(json.dumps({"its": info.its, "reason": info.reason, "seconds": info.seconds_total,
                          "mult_s": info.seconds_mult, "pc_s": info.seconds_pc, "n_mult": info.n_mult,
                          "n_pc": info.n_pc, "launches": s.kernel_launches() - l0,
                          "res": float(np.sqrt((r0 ** 2).sum() + (r1 ** 2).sum())),
                          "hist": info.history[:6] + info.history[-2:]}), flush=True)
    print("mem GB", torch.cuda.max_memory_allocated() / 1e9, torch.cuda.mem_get_info())


if __name__ == "__main__":
    main()
