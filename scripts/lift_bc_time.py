"""Time one ctl_lift_bc at BASELINE config C5 size (P1 on 512 x 512, n_t = 32, CN, per-level Gauss-Newton K_i)
with CUDA events, next to the host non_linear_res_eval that a Picard / Gauss-Newton outer iteration with
inhomogeneous Dirichlet data runs instead when the iterate is not kept on the device.

Prints one JSON line.  The device time is the average over --reps back-to-back launches on the library's stream
(the boundary-column CSR is built on the first, untimed call); the host time is wall clock of one
non_linear_res_eval, the D_v assembly per level included, as that loop pays it."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=512)
    ap.add_argument("--n_t", type=int, default=32)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--host-reps", type=int, default=2)
    args = ap.parse_args()
    import torch
    from synthetic import fem, problems
    from control_b200 import MultiBlockSystem
    from oracle import control as ocontrol
    if not torch.cuda.is_available():
        raise SystemExit("lift_bc_time.py needs a CUDA device")
    n_t = args.n_t
    q = problems.heat_problem(args.nx, n_t, True, beta=1e-2)
    M, bd, tau = q["M"], q["bdofs"], q["tau"]
    n = M.shape[0]
    Dv = fem.nonlinear_diffusion_p1_2d(args.nx, args.nx, 2.0, 2.0)
    times = tau * np.arange(n_t)
    xb, yb = q["coords"][bd, 0], q["coords"][bd, 1]
    g = 0.3 * np.stack([np.cos(xb + t) + 0.5 * yb for t in times])
    rng = np.random.default_rng(0)
    v_old = 0.1 * rng.standard_normal((n_t, n))
    v_old[:, bd] = g
    zeta_old = 0.1 * rng.standard_normal((n_t, n))
    zeta_old[:, bd] = 0.0
    zeta_old[-1] = 0.0
    K = [Dv(v_old[i], True) for i in range(n_t)]
    s = MultiBlockSystem(M, K, n_t=n_t, beta=q["beta"], CN=True, time_interval=q["time_interval"], bc_dofs=bd)
    g_dev = torch.from_numpy(g).to(s.device)
    b = s.new_vector()
    s.lift_bc_device(g_dev, b)                     # builds and uploads the boundary-column CSR
    for _ in range(10):
        s.lift_bc_device(g_dev, b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s.stream)
    for _ in range(args.reps):
        s._lib.ctl_lift_bc(s._h, g_dev.data_ptr(), b.data_ptr(), 0)
    e1.record(s.stream)
    e1.synchronize()
    dev_ms = e0.elapsed_time(e1) / args.reps
    host = []
    for _ in range(args.host_reps):
        t0 = time.perf_counter()
        ocontrol.non_linear_res_eval(M, lambda v, t: Dv(v, True), times, tau, q["beta"], n_t, True, bd, v_old,
                                     zeta_old, v_old[0], q["v_d"], q["f"])
        host.append(time.perf_counter() - t0)
    props = torch.cuda.get_device_properties(s.device)
    power = None
    try:
        import subprocess
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(s.device.index)], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        pass
    print(json.dumps({"config": f"P1 {args.nx}x{args.nx}, n_t={n_t}, CN, per-level Gauss-Newton K_i",
                      "n": n, "n_bc": int(bd.size), "ctl_lift_bc_ms": dev_ms, "reps": args.reps,
                      "host_non_linear_res_eval_s": min(host), "gpu": props.name, "power_limit": power}))
    s.close()


if __name__ == "__main__":
    main()
