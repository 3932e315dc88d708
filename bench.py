#!/usr/bin/env python
"""Benchmark of the all-at-once KKT solve (BASELINE.json: "KKT solve s & SpMM HBM GB/s, heat
control 1024^2 P1 n_t=64").

A step = one complete KKT solve of BASELINE config C2 (2-D heat control, P1 on a
1024 x 1024 mesh of (0,2)^2, n_t = 64, trapezoidal rule, beta = 1e-4, rtol 1e-6) with the
right-hand side resident in HBM.  `value` = seconds per solve (device time, CUDA events, max
over ranks).  `e2e` = the same solve through the public API with HOST buffers (pinned
host -> device copy of b and of the initial guess, device -> host copy of the solution inside
the timed region).  `roofline` = the dominant kernel of the step (fine-level AMG smoother
SpMV of the time sweeps); `roofline_spmm` = the fused time-batched KKT-apply SpMM the metric
names.  `cpu_baseline` = the CPU oracle on a bounded sample of the same workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--ksp minres|fgmres|gmres]
    python bench.py --impl reference ...      # CPU oracle arm (the reference's algorithm)
    python bench.py --dump-outputs DIR ...    # also write the last timed solve's results as DIR/<name>.npy

--dump-outputs writes what a caller of the timed solve receives: the solution blocks (v.npy, zeta.npy; for the Stokes
workload also mu.npy, p.npy) and the residual history of the solve (residual_history.npy), all float64.  A solution
block larger than DUMP_SAMPLE entries is sampled at fixed, seeded (time block, dof) positions in global numbering, so
two builds, or two GPU counts, can be compared entry for entry.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "kkt_solve_time"
UNIT = "s"


def ncu_traffic(key, args):
    """DRAM bytes per launch from the committed ncu --set full capture of the same kernel (only valid for the C2 sizes on
    one GPU; profiles/r02_traffic.json names the capture of every entry)."""
    if args.workload != "heat" or args.nx != 1024 or args.n_t != 64 or args.gpus != 1:
        return None
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))[key]["bytes"]
    except Exception:
        return None


def amg_options(text):
    """"cycles=2,nu=4" -> {"cycles": 2, "nu": 4} (keys of MultiBlockSystem.setup_preconditioner / oracle.amg.DEFAULTS)."""
    out = {}
    for kv in filter(None, (text or "").split(",")):
        k, v = kv.split("=")
        out[k.strip()] = float(v) if "." in v else int(v)
    return out


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for nm, val in zip(names, f[2:]):
                    if val.lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


DUMP_SAMPLE = 1 << 20        # entries kept of each dumped solution block: 8 MB in float64


def sample_blocks(u, parts, dist=None):
    """{name: float64 sample} of the (blocks, n) arrays stored block-major in the rank-local device vector u.
    parts = [(name, offset of the rank's (blocks, n_local) array in u, blocks, n, row_begin, n_local)].  The sample is
    drawn in global (block, dof) numbering and summed over ranks, each entry being owned by exactly one rank."""
    import torch
    out = {}
    for name, offset, blocks, n, rb, nl in parts:
        size = blocks * n
        g = np.arange(size) if size <= DUMP_SAMPLE else \
            np.unique(np.random.default_rng(0).integers(0, size, DUMP_SAMPLE))
        t, j = np.divmod(g, n)
        own = np.flatnonzero((j >= rb) & (j < rb + nl))
        vals = torch.zeros(g.size, dtype=torch.float64, device=u.device)
        vals[torch.from_numpy(own).to(u.device)] = u[torch.from_numpy(offset + t[own] * nl + j[own] - rb).to(u.device)]
        if dist is not None:
            dist.all_reduce(vals)
        out[name] = vals.cpu().numpy()
    return out


def write_outputs(directory, arrays):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), np.asarray(a, dtype=np.float64))


def solver_parameters(ksp, rtol, restart=30):
    return {"linear_solver": ksp, "gmres_restart": restart, "maximum_iterations": 200,
            "relative_tolerance": rtol, "absolute_tolerance": 0.0, "preconditioner": True}


# --------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm in C / OpenMP (oracle/c/pc_omp.c through oracle/fastpc.py) on all host cores.
# One step = ONE complete Krylov iteration at the full size on ALL time blocks (operator apply + preconditioner
# apply + the iteration's vector work), scaled by the iteration count of the solve (its + 1 applications).
# --------------------------------------------------------------------------------------
ITERATION_COUNTS = os.path.join(ROOT, "profiles", "iteration_counts.json")


def problem_key(args):
    key = f"{args.workload}/{args.nx}/{args.n_t}/{args.ksp}/{args.rtol:g}"
    return key + (f"/{args.amg}" if args.amg else "")


def known_iterations(args):
    """Iteration count of the GPU arm on this configuration (same algorithm, same count): measured by this file's
    GPU arm and committed in profiles/iteration_counts.json; --ref_its overrides."""
    if args.ref_its is not None:
        return args.ref_its, "--ref_its"
    rec = n1_expectation(args)
    if rec is not None:
        return int(rec["iterations"]), "profiles/iteration_counts.json (GPU arm)"
    return 15, "assumed (no GPU record for this configuration)"


def n1_expectation(args):
    """Iterations and true residual of this configuration on one GPU (committed record), or None."""
    try:
        rec = json.load(open(ITERATION_COUNTS))[problem_key(args)]
        return rec if isinstance(rec, dict) else {"iterations": int(rec), "kkt_residual": None}
    except Exception:
        return None


class CpuArm:
    def __init__(self, q, args, mode, CN):
        from oracle import fastpc
        self.threads = fastpc.set_threads()      # explicitly all cores: torchrun exports OMP_NUM_THREADS=1
        self.fastpc = fastpc
        self.pc = fastpc.FastPc(q["M"], q["K"], q["tau"], q["beta"], q["n_t"], CN, q["bdofs"],
                                lambda_v_bounds=q["lambda_v_bounds"], mode=mode, amg_params=amg_options(args.amg) or None)
        rng = np.random.default_rng(0)
        N, n = self.pc.N, self.pc.n
        self.x0 = rng.standard_normal((N, n))
        self.x1 = rng.standard_normal((N, n))
        self.x0[:, q["bdofs"]] = 0.0
        self.x1[:, q["bdofs"]] = 0.0
        # vector work of one iteration on the stacked vector: MINRES 2 inner products + 6 updates; (F)GMRES(m)
        # on average m / 2 + 1 of each
        self.n_dots, self.n_axpys = (2, 6) if args.ksp == "minres" else (args.restart // 2 + 1, args.restart // 2 + 1)
        self.iteration()      # untimed: page faults, thread start-up

    def iteration(self):
        t0 = time.perf_counter()
        y0, y1 = self.pc.kkt_apply(self.x0, self.x1)
        t1 = time.perf_counter()
        u0, u1 = self.pc.pc_apply(y0, y1)
        t2 = time.perf_counter()
        self.fastpc.vector_work(u0.reshape(-1), y0.reshape(-1), self.n_dots, self.n_axpys)
        t3 = time.perf_counter()
        return {"kkt_apply_s": t1 - t0, "pc_apply_s": t2 - t1, "vector_s": t3 - t2, "iteration_s": t3 - t0}

    def sample_text(self, args, its, its_source):
        return (f"1 complete {args.ksp} iteration (operator apply + in-built preconditioner apply + the iteration's "
                f"inner products / updates) at the full size on ALL {self.pc.N} time blocks, x{its + 1} applications "
                f"for a solve of {its} iterations [{its_source}]; the reference's algorithm restated in C / OpenMP "
                f"(oracle/c/pc_omp.c, checked against the numpy oracle), AMG set-up once and untimed, "
                f"{self.threads} OpenMP threads on {os.cpu_count()} host cores")


def run_reference(args):
    """--impl reference: the reference's algorithm on the host cores (C / OpenMP port: the real
    Firedrake/PETSc/hypre stack cannot be installed here, DESIGN.md)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from synthetic import problems
    c3 = args.workload == "c3"
    q = problems.heat_problem_3d(args.nx, args.n_t, False) if c3 else problems.heat_problem(args.nx, args.n_t, True)
    mode = "diagonal" if args.ksp == "minres" else "triangular"
    its, its_source = known_iterations(args)
    arm = CpuArm(q, args, mode, not c3)
    times, parts = [], None
    for i in range(args.warmup + args.steps):
        parts = arm.iteration()
        if i >= args.warmup:
            times.append(parts["iteration_s"] * (its + 1))
    val = float(np.mean(times))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": val * 1e3,
            "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": config_dict(args), "iterations": its,
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": arm.threads, "kind": "port",
                             "sample": arm.sample_text(args, its, its_source), **parts},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def inner_text(args):
    a = {"cycles": 3, "nu": 3, **amg_options(args.amg)}
    return (f"{a['cycles']} aggregation-AMG V({a['nu']},{a['nu']}) cycles (the reference: hypre BoomerAMG, "
            f"pc_hypre_boomeramg_max_iter 2, control/control.py:2056-2067)")


def config_dict(args):
    if args.workload == "c3":
        return {"workload": f"C3: 3-D heat control, P1 tetrahedra on the {args.nx}^3 unit-cube mesh, n_t={args.n_t}, "
                            f"backward Euler, beta=1e-4, {args.ksp}({args.restart}) + in-built block lower-triangular "
                            f"preconditioner (the reference's default Krylov parameters, control/control.py:3260-3266), "
                            f"rtol {args.rtol:g}, rows block-partitioned over {args.gpus} GPU(s)",
                "n": (args.nx + 1) ** 3, "n_t": args.n_t, "ksp": args.ksp, "rtol": args.rtol, "amg": args.amg or "library defaults",
                "l2": "Krylov vectors (1.1 GB each) exceed L2; the per-kernel micro-timings rotate through operand sets of "
                      "more than twice the L2 capacity (inputs larger than L2)"}
    return {"workload": f"C2: 2-D heat control, P1 on {args.nx}x{args.nx} mesh of (0,2)^2, n_t={args.n_t}, "
                        f"trapezoidal (CN), beta=1e-4, {args.ksp} + in-built block preconditioner "
                        f"({'block-diagonal SPD variant' if args.ksp == 'minres' else 'block lower-triangular'}), "
                        f"inner solves: {inner_text(args)}, rtol {args.rtol:g}",
            "n": (args.nx + 1) ** 2, "n_t": args.n_t, "ksp": args.ksp, "rtol": args.rtol, "amg": args.amg or "library defaults",
            "l2": "Krylov vectors (1.08 GB each) exceed L2; the per-kernel micro-timings rotate through operand sets of "
                  "more than twice the L2 capacity (inputs larger than L2)"}


def run_stokes(args):
    """--workload stokes: BASELINE config C4 (instationary Stokes control, Taylor-Hood P2-P1 on
    512x512, n_t = 32, CN, FGMRES + pressure-Schur preconditioner), one GPU.  Opt-in: one solve
    takes about a minute, so the default bench stays on config C2."""
    import torch
    from synthetic import problems
    from control_b200.control import build_rhs
    from control_b200.stokes import StokesSystem
    assert args.gpus == 1, "the Stokes path is single-GPU in this round"
    torch.cuda.set_device(0)
    q = problems.stokes_problem(args.nx, args.n_t, True, beta=1.0)
    th = q["th"]
    s = StokesSystem(th["M_v"], th["K_v"], th["B"], th["M_p"], th["K_p"], n_t=q["n_t"], beta=q["beta"], CN=True,
                     time_interval=q["time_interval"], bc_dofs_v=q["bdofs"])
    t0 = time.perf_counter()
    s.setup_preconditioner(lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"])
    setup_s = time.perf_counter() - t0
    N = s.N
    b00, b01 = build_rhs(q["M"], q["K"], q["tau"], q["n_t"], True, q["bdofs"], q["v_d"], q["f"], np.zeros(s.n_v))
    b_np = np.concatenate([b00.ravel(), b01.ravel(), np.zeros(2 * N * s.n_p)])
    b_host = torch.from_numpy(b_np).pin_memory()
    u_host = torch.zeros_like(b_host).pin_memory()
    b_dev = b_host.to(s.device)
    sp_ = {"linear_solver": "fgmres", "gmres_restart": 30, "maximum_iterations": 100, "preconditioner": True,
           "relative_tolerance": args.rtol, "absolute_tolerance": 0.0}

    def solve_resident():
        u = torch.zeros_like(b_dev)
        return s.solve_device(b_dev, u, solver_parameters=sp_), u

    def solve_e2e():
        bd = b_host.to(s.device, non_blocking=True)
        ud = u_host.to(s.device, non_blocking=True)
        info = s.solve_device(bd, ud, solver_parameters=sp_)
        u_host.copy_(ud, non_blocking=True)
        torch.cuda.synchronize()
        return info

    for _ in range(args.warmup):
        solve_resident()
    torch.cuda.synchronize()
    l0 = s.kernel_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(0) as clocks:
        ev0.record()
        for _ in range(args.steps):
            info, u_last = solve_resident()
        ev1.record()
        torch.cuda.synchronize()
    launches = s.kernel_launches() - l0
    value = ev0.elapsed_time(ev1) * 1e-3 / args.steps
    if args.dump_outputs:
        N, n_v, n_p = s.N, s.n_v, s.n_p
        parts = [("v", 0, N, n_v, 0, n_v), ("zeta", N * n_v, N, n_v, 0, n_v),
                 ("mu", 2 * N * n_v, N, n_p, 0, n_p), ("p", 2 * N * n_v + N * n_p, N, n_p, 0, n_p)]
        write_outputs(args.dump_outputs, {**sample_blocks(u_last, parts), "residual_history": info.history})
    r0, r1 = s.to_host_blocks(b_dev - s.apply(u_last))
    r0[:, q["bdofs"]] = 0.0
    r1 = r1 - r1.mean(axis=1, keepdims=True)
    t0 = time.perf_counter()
    solve_e2e()
    e2e_s = time.perf_counter() - t0
    peak, peak_src = measured_peak()
    div = s.time_divergence_products(20)
    micro = s.velocity.micro_benchmarks(flush_l2=True)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": value * 1e3, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"C4: instationary Stokes control, Taylor-Hood P2-P1 on {args.nx}x{args.nx} mesh of "
                                   f"(0,2)^2, n_t={args.n_t}, trapezoidal (CN), beta=1, FGMRES(30) + in-built "
                                   f"pressure-Schur preconditioner (5 inner GMRES iterations), rtol {args.rtol:g}",
                       "n_v": s.n_v, "n_p": s.n_p, "n_t": args.n_t, "rtol": args.rtol,
                       "l2": "Krylov vectors (1.2 GB each) exceed L2"},
            "iterations": info.its, "converged_reason": info.reason,
            "kkt_residual": float(np.sqrt((r0 ** 2).sum() + (r1 ** 2).sum())),
            "rel_residual": info.rnorm / info.ref_norm if info.ref_norm else None,
            "setup_s": setup_s, "pc_apply_ms": info.seconds_pc / max(1, info.n_pc) * 1e3,
            "operator_apply_ms": info.seconds_mult / max(1, info.n_mult) * 1e3, "peak_source": peak_src,
            "roofline": {"kernel": "sell_cheb_kernel, velocity AMG level 0 (smoother step of the time sweeps)",
                         "bound": "hbm", "achieved": micro["cheb_bytes"] / micro["cheb_ms"] / 1e6, "peak": peak,
                         "unit": "GB/s", "frac": micro["cheb_bytes"] / micro["cheb_ms"] / 1e6 / peak, "traffic": None,
                         "alg_bytes_per_launch": micro["cheb_bytes"], "ms_per_launch": micro["cheb_ms"],
                         "how": "CUDA events per launch, L2 flushed between launches"},
            "roofline_spmm": {"kernel": "panel_spmm_kernel (tau B X on one time panel)", "bound": "hbm",
                              "achieved": div["B_bytes"] / div["B_ms"] / 1e6, "peak": peak, "unit": "GB/s",
                              "frac": div["B_bytes"] / div["B_ms"] / 1e6 / peak, "traffic": None,
                              "alg_bytes_per_launch": div["B_bytes"], "ms_per_launch": div["B_ms"],
                              "transposed": {"achieved": div["BT_bytes"] / div["BT_ms"] / 1e6,
                                             "frac": div["BT_bytes"] / div["BT_ms"] / 1e6 / peak,
                                             "alg_bytes_per_launch": div["BT_bytes"], "ms_per_launch": div["BT_ms"]},
                              "how": "CUDA events around 20 back-to-back launches (panels exceed L2)"},
            "e2e": {"value": e2e_s, "unit": UNIT, "h2d_bytes_per_step": 2 * b_host.numel() * 8,
                    "d2h_bytes_per_step": b_host.numel() * 8},
            "gpu_launches": int(launches), "clocks": clocks.summary(), "kernels": micro}
    print(json.dumps(line), flush=True)
    s.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="heat", choices=["heat", "c3", "stokes"],
                    help="heat = config C2 (default, the metric's configuration); c3 = config C3 (3-D, backward Euler, "
                         "the configuration BASELINE names for 8 GPUs); stokes = config C4 (opt-in)")
    ap.add_argument("--restart", type=int, default=30)
    ap.add_argument("--nx", type=int, default=1024)
    ap.add_argument("--n_t", type=int, default=64)
    ap.add_argument("--ksp", default="minres", choices=["minres", "fgmres", "gmres"])
    ap.add_argument("--rtol", type=float, default=1e-6)
    ap.add_argument("--ref_its", type=int, default=None,
                    help="iteration count the reference arm scales its one timed iteration by (default: the GPU arm's "
                         "measured count for this configuration, profiles/iteration_counts.json)")
    ap.add_argument("--amg", default=None,
                    help="inner-solver parameters, e.g. cycles=2,nu=4 (both arms); default: cycles=2,nu=4 for the "
                         "block-diagonal MINRES configuration of C2 -- two cycles as in the reference, 15 iterations as "
                         "with the library default of three V(3,3) cycles (profiles/r02_amg_param_sweep.txt) -- and the "
                         "library defaults otherwise")
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--no_alt", action="store_true", help="skip the FGMRES + triangular PC side measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the solution blocks (a fixed, seeded sample of at most DUMP_SAMPLE entries each) and "
                         "the residual history of the last timed solve as DIR/<name>.npy, float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the timed GPU solve (--impl b200)")
    if args.workload == "c3":
        # config C3 and the reference's default Krylov parameters (control/control.py:3260-3266): GMRES(10)
        if args.nx == 1024 and args.n_t == 64:
            args.nx, args.n_t = 128, 32
        if args.ksp == "minres":
            args.ksp, args.restart = "gmres", 10
    if args.amg is None:
        args.amg = "cycles=2,nu=4" if (args.workload == "heat" and args.ksp == "minres") else ""
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "stokes":
        if args.nx == 1024 and args.n_t == 64:          # the heat defaults: switch to config C4's
            args.nx, args.n_t = 512, 32
        return run_stokes(args)

    import torch
    from synthetic import problems
    from control_b200 import MultiBlockSystem, _lib as L
    from control_b200.control import build_rhs

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    c3 = args.workload == "c3"
    q = problems.heat_problem_3d(args.nx, args.n_t, False) if c3 else problems.heat_problem(args.nx, args.n_t, True)
    CN = not c3
    mode = "diagonal" if args.ksp == "minres" else "triangular"
    s = MultiBlockSystem(q["M"], q["K"], n_t=q["n_t"], beta=q["beta"], CN=CN,
                         time_interval=q["time_interval"], bc_dofs=q["bdofs"], device=local_rank,
                         rank=rank, world=world)
    if world > 1:
        s.init_comm(dist)
    t0 = time.perf_counter()
    s.setup_preconditioner(lambda_v_bounds=q["lambda_v_bounds"], mode=mode, **amg_options(args.amg))
    setup_s = time.perf_counter() - t0
    b0, b1 = build_rhs(q["M"], q["K"], q["tau"], q["n_t"], CN, q["bdofs"], q["v_d"], q["f"], np.zeros(s.n))
    rows = slice(s.row_begin, s.row_begin + s.n_local)
    b0, b1 = np.ascontiguousarray(b0[:, rows]), np.ascontiguousarray(b1[:, rows])
    sp_ = solver_parameters(args.ksp, args.rtol, args.restart)
    b_dev = s.to_device(b0, b1)
    b_host = torch.from_numpy(np.concatenate([b0.ravel(), b1.ravel()])).pin_memory()
    u_host = torch.zeros_like(b_host).pin_memory()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def solve_resident():
        u = s.new_vector()
        return s.solve_device(b_dev, u, solver_parameters=sp_, pc="builtin"), u

    def solve_e2e():
        u_host.zero_()
        bd = b_host.to(s.device, non_blocking=True)
        ud = u_host.to(s.device, non_blocking=True)
        info = s.solve_device(bd, ud, solver_parameters=sp_, pc="builtin")
        u_host.copy_(ud, non_blocking=True)
        torch.cuda.synchronize()
        return info

    for _ in range(args.warmup):
        solve_resident()
    # ---- timed region: exactly `steps` solves, device time, max over ranks
    barrier()
    l0 = s.kernel_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    infos = []
    with ClockSampler(local_rank) as clocks:
        ev0.record()
        for _ in range(args.steps):
            info, u_last = solve_resident()
            infos.append(info)
        ev1.record()
        barrier()
    launches = s.kernel_launches() - l0
    total_s = max_over_ranks(ev0.elapsed_time(ev1) * 1e-3)
    value = total_s / args.steps
    res_norm = s.residual_norm(b_dev, u_last)
    if args.dump_outputs:
        blocks = (s.N, s.n, s.row_begin, s.n_local)
        out = sample_blocks(u_last, [("v", 0, *blocks), ("zeta", s.N * s.n_local, *blocks)], dist)
        if rank == 0:
            write_outputs(args.dump_outputs, {**out, "residual_history": infos[-1].history})

    # ---- end to end through the public API with host buffers
    solve_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        solve_e2e()
    barrier()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / args.steps)
    nbytes = b_host.numel() * 8

    info = infos[-1]
    # ---- roofline: KKT-apply SpMM, live over the timed region (events around every apply)
    peak, peak_src = measured_peak()
    n, N, nnz = s.n_local, s.N, int(q["M"].nnz * s.n_local / s.n)
    spmm_bytes = 32.0 * n * N + 20.0 * nnz + 4.0 * (n + 1)
    spmm_ms = sum(i.seconds_mult for i in infos) / sum(i.n_mult for i in infos) * 1e3
    roof_spmm = {"kernel": "kkt_apply_staged_kernel (fused time-batched KKT SpMM)", "bound": "hbm",
                 "achieved": spmm_bytes / spmm_ms / 1e6, "peak": peak, "unit": "GB/s",
                 "frac": spmm_bytes / spmm_ms / 1e6 / peak, "traffic": ncu_traffic("kkt_apply_C2", args),
                 "alg_bytes_per_launch": spmm_bytes, "ms_per_launch": spmm_ms,
                 "how": "CUDA events around every apply inside the timed solves"}
    # ---- roofline: dominant kernel of the step = fine-level smoother SpMV of the AMG sweeps
    micro = s.micro_benchmarks(reps=20, flush_l2=True) if hasattr(s, "micro_benchmarks") else None
    roof = roof_spmm
    if micro:
        roof = {"kernel": "sell_cheb_kernel, AMG level 0 (smoother step of the time sweeps)", "bound": "hbm",
                "achieved": micro["cheb_bytes"] / micro["cheb_ms"] / 1e6, "peak": peak, "unit": "GB/s",
                "frac": micro["cheb_bytes"] / micro["cheb_ms"] / 1e6 / peak,
                "traffic": ncu_traffic("sell_cheb_kernel_level0_C2", args),
                "alg_bytes_per_launch": micro["cheb_bytes"], "ms_per_launch": micro["cheb_ms"],
                "how": "CUDA events around 20 launches on the library's stream, every launch on its own operand set, "
                       "the sets rotating through > 2 x L2 (inputs larger than L2); alg_bytes = the bytes of the exact "
                       "compressed matrix format in use + 5 vectors; SURVEY 8(d)'s CSR model of the same product "
                       "(12 nnz + 40 n) is in survey_model",
                "survey_model": {"alg_bytes_per_launch": 12.0 * nnz + 40.0 * n,
                                 "achieved": (12.0 * nnz + 40.0 * n) / micro["cheb_ms"] / 1e6,
                                 "frac": (12.0 * nnz + 40.0 * n) / micro["cheb_ms"] / 1e6 / peak},
                "inner_solve": {"ms": micro["inner_solve_ms"], "alg_bytes": micro["inner_solve_bytes"],
                                "kernels": micro["inner_solve_kernels"],
                                "achieved": micro["inner_solve_bytes"] / micro["inner_solve_ms"] / 1e6,
                                "frac": micro["inner_solve_bytes"] / micro["inner_solve_ms"] / 1e6 / peak}}
    pc_s = sum(i.seconds_pc for i in infos) / max(1, sum(i.n_pc for i in infos))

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": value * 1e3, "higher_is_better": False,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(args),
            "iterations": info.its, "converged_reason": info.reason, "kkt_residual": res_norm,
            "rel_residual": info.rnorm / info.ref_norm if info.ref_norm else None,
            "setup_s": setup_s, "pc_apply_ms": pc_s * 1e3, "kkt_apply_ms": spmm_ms,
            "peak_source": peak_src,
            "roofline": roof, "roofline_spmm": roof_spmm,
            "e2e": {"value": e2e_s, "unit": UNIT, "h2d_bytes_per_step": 2 * nbytes, "d2h_bytes_per_step": nbytes},
            "gpu_launches": int(launches), "clocks": clocks.summary()}
    exp = n1_expectation(args)
    if exp is not None:
        # the same solve on any number of GPUs must reproduce the one-GPU record: identical iteration count, true
        # residual equal up to the summation order of the partitioned products
        res_exp = exp.get("kkt_residual")
        line["parity_vs_1gpu"] = {"expected_iterations": exp["iterations"], "iterations_match": info.its == exp["iterations"],
                                  "expected_kkt_residual": res_exp,
                                  "kkt_residual_rel_diff": (abs(res_norm - res_exp) / res_exp) if res_exp else None,
                                  "source": "profiles/iteration_counts.json"}
    if micro:
        line["kernels"] = micro
    if args.ksp == "minres" and not args.no_alt:
        # the reference-faithful mode next to the configuration BASELINE.json names: block
        # lower-triangular in-built preconditioner + FGMRES(30) (control/control.py:1943-2440)
        s.setup_preconditioner(lambda_v_bounds=q["lambda_v_bounds"], mode="triangular")      # library defaults: 3 V(3,3) cycles
        sp2 = solver_parameters("fgmres", args.rtol)
        for _ in range(2):
            u2 = s.new_vector()
            barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            i2 = s.solve_device(b_dev, u2, solver_parameters=sp2, pc="builtin")
            a1.record()
            barrier()
        line["alt_fgmres_triangular"] = {"value": max_over_ranks(a0.elapsed_time(a1) * 1e-3), "unit": UNIT,
                                         "amg": "cycles=3,nu=3 (library defaults)", "iterations": i2.its, "converged_reason": i2.reason,
                                         "kkt_residual": s.residual_norm(b_dev, u2)}
    if rank == 0 and not args.no_cpu_baseline:
        t0 = time.perf_counter()
        arm = CpuArm(q, args, mode, CN)
        parts = arm.iteration()
        line["cpu_baseline"] = {"value": parts["iteration_s"] * (info.its + 1), "unit": UNIT, "cores": arm.threads,
                                "kind": "port", "sample": arm.sample_text(args, info.its, "this run's GPU arm"),
                                **parts, "wall_s": time.perf_counter() - t0}
        del arm
    if rank == 0:
        print(json.dumps(line), flush=True)
    s.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
