"""Time of one AMG inner solve at config C2 (warm, back to back) and of the level-0 kernels -- for A/B experiments
between builds, or between the keyword arguments of setup_preconditioner (argv[2], JSON)."""
import json, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from synthetic import problems
from control_b200 import MultiBlockSystem
nx = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
kw = json.loads(sys.argv[2]) if len(sys.argv) > 2 else {}
q = problems.heat_problem(nx, 64, True)
s = MultiBlockSystem(q["M"], q["K"], n_t=64, beta=q["beta"], CN=True, time_interval=q["time_interval"], bc_dofs=q["bdofs"])
t0 = time.perf_counter()
s.setup_preconditioner(lambda_v_bounds=q["lambda_v_bounds"], **kw)
setup = time.perf_counter() - t0
a = s.micro_benchmarks(reps=30, flush_l2=False)
b = s.micro_benchmarks(reps=30, flush_l2=True)
env = {k: v for k, v in os.environ.items() if k.startswith("CTL_")}
print(json.dumps({"env": env, "kw": kw, "nx": nx, "setup_s": round(setup, 3), "inner_solve_ms": round(a["inner_solve_ms"], 4),
                  "kernels": a["inner_solve_kernels"], "cheb_warm_us": round(a["cheb_ms"] * 1e3, 2),
                  "cheb_flushed_us": round(b["cheb_ms"] * 1e3, 2), "resid_warm_us": round(a["residual_ms"] * 1e3, 2),
                  "cheb_bytes": a["cheb_bytes"], "inner_bytes": a["inner_solve_bytes"]}), flush=True)
