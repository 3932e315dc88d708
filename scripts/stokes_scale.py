"""Strong scaling of the instationary Stokes control solve (BASELINE config C4 by default: Taylor-Hood P2-P1 on 512x512,
n_t = 32, CN, FGMRES(30) + the in-built pressure-Schur preconditioner), row-partitioned over the ranks of torchrun:

    python scripts/stokes_scale.py                                   # 1 GPU
    python scripts/stokes_scale.py --block-size 2                    # 1 GPU, block-scalar velocity sweeps
    torchrun --nproc-per-node 4 scripts/stokes_scale.py --ref-its 18 # 4 GPUs, parity against the 1-GPU count

Rank 0 prints one JSON line (and appends it to --out when given): the card name and power limit, outer iterations,
solve and set-up seconds, the true residual ||b - A u|| / ||b|| (velocity Dirichlet rows and pressure means removed,
as the solve's projection does), parity against --ref-its, and per rank the ghost rows of the two divergence-product
exchange plans, the time of one tau B X / Y += tau B^T X panel product including its exchange, and the GPU memory in
use after set-up.  Nothing is written to the repository tree."""
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


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=512)
    ap.add_argument("--n_t", type=int, default=32)
    ap.add_argument("--beta", type=float, default=1.0)
    ap.add_argument("--rtol", type=float, default=1e-6)
    ap.add_argument("--restart", type=int, default=30)
    ap.add_argument("--max_it", type=int, default=100)
    ap.add_argument("--block-size", type=int, default=1, help="velocity block size (2: block-scalar sweeps, one GPU)")
    ap.add_argument("--ref-its", type=int, default=None, help="outer iterations of the one-GPU run, for the parity flag")
    ap.add_argument("--reps", type=int, default=20, help="launches per divergence-product timing")
    ap.add_argument("--out", default=None, help="append the JSON line to this file")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    dev = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
    from control_b200 import partition
    from control_b200.control import build_rhs
    from control_b200.stokes import StokesSystem
    from synthetic import problems

    def gather(x):
        if dist is None:
            return [x]
        parts = [None] * world
        dist.all_gather_object(parts, x)
        return parts

    def allsum(v):
        t = torch.tensor(v, dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t)
        return t.cpu().numpy()

    CN = True
    t0 = time.time()
    q = problems.stokes_problem(args.nx, args.n_t, CN, beta=args.beta)
    th = q["th"]
    assemble_s = time.time() - t0
    kw = dict(rank=rank, world=world) if world > 1 else {}
    s = StokesSystem(th["M_v"], th["K_v"], th["B"], th["M_p"], th["K_p"], n_t=q["n_t"], beta=q["beta"], CN=CN,
                     time_interval=q["time_interval"], bc_dofs_v=q["bdofs"], velocity_block_size=args.block_size, **kw)
    s.init_comm(dist)
    torch.cuda.synchronize()
    t0 = time.time()
    s.setup_preconditioner(lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"])
    torch.cuda.synchronize()
    setup_s = time.time() - t0
    free, total = torch.cuda.mem_get_info()
    mem_gb = (total - free) / 1e9
    N, rv, rp = s.N, s.velocity_rows, s.pressure_rows
    b00, b01 = build_rhs(q["M"], q["K"], q["tau"], q["n_t"], CN, q["bdofs"], q["v_d"], q["f"], np.zeros(s.n_v))
    b = s.to_device(np.ascontiguousarray(np.concatenate([b00, b01])[:, rv]), np.zeros((2 * N, s.n_p_local)))
    del b00, b01
    sp_ = {"linear_solver": "fgmres", "gmres_restart": args.restart, "maximum_iterations": args.max_it,
           "preconditioner": True, "relative_tolerance": args.rtol, "absolute_tolerance": 0.0}
    u = torch.zeros_like(b)
    info = s.solve_device(b, u, solver_parameters=sp_)
    # true residual: constrained velocity rows zero, per-block pressure means (global) removed
    r0, r1 = s.to_host_blocks(b - s.apply(u))
    b0, b1 = s.to_host_blocks(b)
    local_bc = q["bdofs"][(q["bdofs"] >= rv.start) & (q["bdofs"] < rv.stop)] - rv.start
    r0[:, local_bc] = 0.0
    sums = allsum(np.concatenate([[(r0 ** 2).sum(), (b0 ** 2).sum() + (b1 ** 2).sum()], r1.sum(axis=1),
                                  (r1 ** 2).sum(axis=1)]))
    means = sums[2:2 + 2 * N] / s.n_p
    res2 = sums[0] + (sums[2 + 2 * N:] - s.n_p * means ** 2).sum()
    rel_res = float(np.sqrt(max(res2, 0.0) / sums[1]))
    div = s.time_divergence_products(args.reps)
    B = th["B"].tocsr()
    B.sort_indices()
    BT = B.T.tocsr()
    ghosts_B = partition.halo_plan(B.indptr, B.indices, world, rank, n_cols=B.shape[1])["ghosts"].size
    ghosts_BT = partition.halo_plan(BT.indptr, BT.indices, world, rank, n_cols=BT.shape[1])["ghosts"].size
    per_rank = gather(dict(rank=rank, n_v_local=s.n_v_local, n_p_local=s.n_p_local, ghost_rows_B=int(ghosts_B),
                           ghost_rows_BT=int(ghosts_BT), B_ms=round(div["B_ms"], 4), BT_ms=round(div["BT_ms"], 4),
                           mem_in_use_gb=round(mem_gb, 2)))
    if rank == 0:
        rec = {"card": card(), "gpus": world, "block_size": args.block_size, "pc_block_size": s.velocity.pc_block_size,
               "nx": args.nx, "n_t": args.n_t, "n_v": s.n_v, "n_p": s.n_p, "its": info.its, "reason": info.reason,
               "solve_s": round(info.seconds_total, 3), "pc_s": round(info.seconds_pc, 3),
               "setup_s": round(setup_s, 2), "assemble_s": round(assemble_s, 1), "true_rel_residual": rel_res,
               "parity_its": None if args.ref_its is None else info.its == args.ref_its, "ranks": per_rank}
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")
    s.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
