"""Wall time per outer iteration of the Navier-Stokes Picard loop, host loop against device loop, and the time of one
ctl_stokes_nonlinear_residual at BASELINE config C4 size.

Part 1: Control.Instationary.incompressible_non_linear_solve on the lid-driven cavity of the reference's
Navier-Stokes tests (vector Q2 - Q1, nu = 1/100, time-dependent lid data; tests/kat.py) with device_loop=False and
device_loop=True, on the same GPU, one after the other.  Every call below is timed exclusively (a call inside another
timed call is not counted twice) and the time is split into
  assembly    the caller-side forward forms D_v_i / D_p_i (what Firedrake assembles in the reference)
  residual    host non_linear_res_eval (host loop; the B / B^T products of res_eval are in "other") or
              ctl_stokes_nonlinear_residual (device loop)
  pc_setup    StokesSystem.setup_preconditioner
  solve       StokesSystem.solve_device (ends in a device synchronise)
  other       the rest: right-hand sides, lifting, host <-> device copies, vector updates
and reported per outer iteration (loop wall time / outer iterations; the initial residual is included).

Part 2: ctl_stokes_nonlinear_residual alone at C4 size (Taylor-Hood P2 - P1 on 512 x 512, n_t = 32, CN), CUDA events
around --reps back-to-back calls on the library's stream after warm-up.  The outer vectors (1.2 GB each) exceed L2.
The byte model counts every array once per pass of the implementation that touches it: two layout conversions in, the
fused KKT apply, two B^T and two B panel products, the residual/norm epilogue, one conversion out.

Prints JSON lines; the last one carries the card name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

HBM_BYTES_PER_S = 7.7e12       # HGX B200 data sheet, one GPU


class ExclusiveTimers:
    """Wraps methods and callables; time spent in nested wrapped calls goes to the inner category only."""

    def __init__(self):
        self.t = {}
        self._stack = []
        self._undo = []

    def wrap_fn(self, fn, cat):
        def inner(*a, **k):
            t0 = time.perf_counter()
            self._stack.append(0.0)
            try:
                return fn(*a, **k)
            finally:
                dt = time.perf_counter() - t0
                nested = self._stack.pop()
                self.t[cat] = self.t.get(cat, 0.0) + dt - nested
                if self._stack:
                    self._stack[-1] += dt
        return inner

    def wrap_method(self, cls, name, cat):
        orig = getattr(cls, name)
        setattr(cls, name, self.wrap_fn(orig, cat))
        self._undo.append((cls, name, orig))

    def restore(self):
        for cls, name, orig in reversed(self._undo):
            setattr(cls, name, orig)
        self._undo = []


def run_loop(q, nx, device_loop, max_iter):
    from control_b200 import Control
    from control_b200.stokes import StokesSystem
    n_t = q["n_t"]
    T = ExclusiveTimers()
    D_v, D_p = T.wrap_fn(q["D_v"], "assembly"), T.wrap_fn(q["D_p"], "assembly")

    def level(t):
        return int(round(t / q["tau"]))
    c = Control.Instationary(q["M"], lambda v_i, t, gn: D_v(v_i, t),
                             desired_state=lambda t: (q["v_d"][level(t)], q["v_hat"][level(t)]), beta=q["beta"],
                             n_t=n_t, CN=True, time_interval=q["time_interval"], bc_dofs=q["bdofs"],
                             bc_values=lambda t: q["bc_values"][level(t)])
    space_p = dict(B=q["B"], M_p=q["sq"]["M_p"], K_p=q["sq"]["L_p"], forward_matrix_p=lambda v_i, t, gn: D_p(v_i, t))
    T.wrap_method(Control.Instationary, "non_linear_res_eval", "residual")
    T.wrap_method(StokesSystem, "nonlinear_residual", "residual")
    T.wrap_method(StokesSystem, "setup_preconditioner", "pc_setup")
    T.wrap_method(StokesSystem, "solve_device", "solve")
    sp_ = {"linear_solver": "fgmres", "maximum_iterations": 200, "relative_tolerance": 1e-6, "absolute_tolerance": 0.0,
           "monitor_convergence": False}
    try:
        t0 = time.perf_counter()
        k = c.incompressible_non_linear_solve("constant", space_p=space_p, solver_parameters=sp_,
                                              lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"],
                                              max_non_linear_iter=max_iter, print_error_non_linear=False,
                                              device_loop=device_loop)
        wall = time.perf_counter() - t0
    finally:
        T.restore()
    out = {"loop": "device" if device_loop else "host", "nx": nx, "n_t": n_t, "n_v": int(q["M"].shape[0]),
           "n_p": int(q["sq"]["M_p"].shape[0]), "outer_iterations": k, "inner_iterations": list(c.inner_iterations),
           "history": list(c.non_linear_history), "wall_s": wall, "per_iteration_s": wall / max(k, 1)}
    parts = {cat: T.t.get(cat, 0.0) / max(k, 1) for cat in ("assembly", "residual", "pc_setup", "solve")}
    parts["other"] = out["per_iteration_s"] - sum(parts.values())
    out["per_iteration_breakdown_s"] = parts
    c.close()
    return out


def residual_c4(nx, n_t, reps):
    import torch
    from synthetic import problems
    from control_b200.stokes import StokesSystem
    q = problems.stokes_problem(nx, n_t, True, beta=1.0)
    th = q["th"]
    s = StokesSystem(th["M_v"], th["K_v"], th["B"], th["M_p"], th["K_p"], n_t=q["n_t"], beta=q["beta"], CN=True,
                     time_interval=q["time_interval"], bc_dofs_v=q["bdofs"])
    N, n_v, n_p, ld = s.N, s.n_v, s.n_p, s.velocity.ld
    gen = torch.Generator(device=s.device).manual_seed(0)
    b = torch.randn(s.vec_len(), dtype=torch.float64, device=s.device, generator=gen)
    x = torch.randn(s.vec_len(), dtype=torch.float64, device=s.device, generator=gen)
    r = s.new_vector()
    for _ in range(3):
        s.nonlinear_residual(b, x, r)
    torch.cuda.synchronize()
    import ctypes as C
    out = C.c_double()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s.velocity.stream)
    for _ in range(reps):
        s._lib.ctl_stokes_nonlinear_residual(s._s, b.data_ptr(), x.data_ptr(), r.data_ptr(), C.byref(out))
    e1.record(s.velocity.stream)
    e1.synchronize()
    ms = e0.elapsed_time(e1) / reps
    # byte model (see the module docstring); panels are n x ld doubles, block-major vectors 2 N n doubles per space
    nnz_v, nnz_B = th["M_v"].nnz, th["B"].nnz
    K_sym = abs(th["K_v"] - th["K_v"].T).max() == 0.0
    L_bm = 2 * N * (n_v + n_p)
    L_tf = 2 * ld * (n_v + n_p)
    pv, pp = n_v * ld, n_p * ld
    d = 8
    bytes_ = {
        "layout_in": d * 2 * (L_bm + L_tf),                                                 # b and x
        "kkt_apply": d * 2 * 2 * pv + 4 * (n_v + 1) + nnz_v * (4 + d + d * (1 if K_sym else 2)),
        "BT_products": 2 * (12 * nnz_B + 4 * (n_v + 1) + d * (pp + 2 * pv)),
        "B_products": 2 * (12 * nnz_B + 4 * (n_p + 1) + d * (pv + 2 * pp)),
        "epilogue": d * (3 * 2 * pv + 2 * pp) + n_v,
        "layout_out": d * (L_tf + L_bm),
    }
    total = sum(bytes_.values())
    s.close()
    return {"config": f"C4: Taylor-Hood P2-P1 {nx}x{nx}, n_t={n_t}, CN, time-independent K_v", "n_v": n_v, "n_p": n_p,
            "N": N, "ld": ld, "outer_vector_GB": L_bm * 8 / 1e9, "ctl_stokes_nonlinear_residual_ms": ms, "reps": reps,
            "model_bytes": bytes_, "model_GB": total / 1e9, "achieved_TB_per_s": total / (ms * 1e-3) / 1e12,
            "fraction_of_hbm_7.7TBps": total / (ms * 1e-3) / HBM_BYTES_PER_S}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="64,128", help="comma list of cavity cells per side")
    ap.add_argument("--n_t", type=int, default=10)
    ap.add_argument("--max-iter", type=int, default=10)
    ap.add_argument("--c4-nx", type=int, default=512)
    ap.add_argument("--c4-n_t", type=int, default=32)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--skip-c4", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ns_loop_time.py needs a CUDA device")
    import kat
    for nx in [int(v) for v in args.sizes.split(",") if v]:
        q = kat.reference_navier_stokes_problem(True, nx=nx, n_t=args.n_t)
        for device_loop in (False, True):
            print(json.dumps(run_loop(q, nx, device_loop, args.max_iter)), flush=True)
    if not args.skip_c4:
        print(json.dumps(residual_c4(args.c4_nx, args.c4_n_t, args.reps)), flush=True)
    power = None
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True,
                               timeout=30).stdout.strip()
    except Exception:
        pass
    print(json.dumps({"gpu": torch.cuda.get_device_name(), "name_power_limit": power}))


if __name__ == "__main__":
    main()
