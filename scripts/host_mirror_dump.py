"""Runs every scenario of tests/test_host_mirror.py on the CPU -- the ``Control`` drivers with the oracle-backed
stand-in systems of that test module -- with every print switch on, and writes what the drivers leave behind:
``non_linear_history``, ``inner_iterations``, ``_v``, ``_zeta``, ``_p`` and ``_mu`` of each scenario to ``<out>.npz``
and the captured standard output to ``<out>.txt``.  Two runs of different versions of the host layer compare with
``--compare a b``: arrays bitwise, output line by line.

    python scripts/host_mirror_dump.py /tmp/before
    python scripts/host_mirror_dump.py /tmp/after
    python scripts/host_mirror_dump.py --compare /tmp/before /tmp/after
"""
import argparse
import contextlib
import io
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import kat  # noqa: E402
from synthetic import fem  # noqa: E402
from test_host_mirror import SP, FakeMultiBlockSystem, FakeStokesSystem, _stationary_stokes_kat  # noqa: E402

FIELDS = ("non_linear_history", "inner_iterations", "_v", "_zeta", "_p", "_mu")


def _stand_ins():
    import control_b200.control as cc
    import control_b200.stationary as cs
    import control_b200.stokes as cst
    cc.MultiBlockSystem = FakeMultiBlockSystem
    cs.MultiBlockSystem = FakeMultiBlockSystem
    cst.StokesSystem = FakeStokesSystem
    from control_b200 import Control
    return Control


def _level(tau):
    return lambda t: int(round(t / tau))


def scenarios(Control):
    """(name, thunk returning the driver instance) in the order of the test module."""
    def stationary_heat():
        nx = 8
        M, L, coords, bd = fem.assemble_p1_2d(nx, nx, 1.0, 1.0)
        x, y = coords[:, 0], coords[:, 1]
        v_hat = np.sin(np.pi * x) * np.sin(np.pi * y) * np.exp(x + y)
        g = np.cos(3.0 * x[bd]) + y[bd]
        f = M @ (x * y)
        c = Control.Stationary(M, (L + 2.0 * M).tocsr(), desired_state=lambda: (M @ v_hat, v_hat), force_f=lambda: f,
                               beta=1e-2, bc_dofs=bd, bc_values=g)
        c.linear_solve(solver_parameters=SP, lambda_v_bounds=(0.5, 2.0), print_error=True)
        out = [("stationary_linear", c)]
        D = fem.nonlinear_diffusion_p1_2d(nx, nx, 1.0, 1.0)
        for gn in (False, True):
            c = Control.Stationary(M, D, desired_state=lambda: (M @ v_hat, v_hat), beta=1e-2, Gauss_Newton=gn, bc_dofs=bd)
            c.non_linear_solve(solver_parameters=SP, lambda_v_bounds=(0.5, 2.0), max_non_linear_iter=30,
                               print_error_linear=True, print_error_non_linear=True)
            out.append((f"stationary_non_linear_gn{int(gn)}", c))
        return out

    def convection_diffusion(CN):
        q = kat.mms_convection_diffusion_problem(4, 12, CN)
        lv = _level(q["tau"])
        c = Control.Instationary(q["M"], lambda v_i, t, gn: q["K_levels"][lv(t)],
                                 desired_state=lambda t: (q["v_d"][lv(t)], q["v_hat"][lv(t)]),
                                 force_f=lambda t: q["f"][lv(t)], beta=q["beta"], n_t=q["n_t"], CN=CN,
                                 time_interval=q["time_interval"], bc_dofs=q["bdofs"],
                                 bc_values=lambda t: q["bc_values"][lv(t)], initial_condition=q["v_0"])
        c.linear_solve(solver_parameters=SP, lambda_v_bounds=(0.5, 2.0), print_error=True)
        return [(f"convection_diffusion_cn{int(CN)}", c)]

    def navier_stokes(CN):
        q = kat.reference_navier_stokes_problem(CN, nx=4, n_t=6)
        sq, lv = q["sq"], _level(q["tau"])
        c = Control.Instationary(q["M"], lambda v_i, t, gn: q["D_v"](v_i, t),
                                 desired_state=lambda t: (q["v_d"][lv(t)], q["v_hat"][lv(t)]), beta=q["beta"],
                                 n_t=q["n_t"], CN=CN, time_interval=q["time_interval"], bc_dofs=q["bdofs"],
                                 bc_values=lambda t: q["bc_values"][lv(t)])
        space_p = dict(B=q["B"], M_p=sq["M_p"], K_p=sq["L_p"], forward_matrix_p=lambda v_i, t, gn: q["D_p"](v_i, t))
        c.incompressible_non_linear_solve("constant", space_p=space_p, solver_parameters=dict(SP, relative_tolerance=1e-8),
                                          lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"],
                                          print_error_linear=True, print_error_non_linear=True)
        return [(f"navier_stokes_cn{int(CN)}", c)]

    def stationary_stokes():
        k = _stationary_stokes_kat()
        sp_ = {"linear_solver": "fgmres", "fgmres_restart": 10, "maximum_iterations": 500, "relative_tolerance": 1e-14,
               "absolute_tolerance": 1e-14}
        c = Control.Stationary(k["M"], k["K"], beta=k["beta"], bc_dofs=k["bd"])
        space_p = dict(B=k["B"], M_p=k["Mp"], K_p=k["Lp"], forward_matrix_p=k["D_p"])
        c.incompressible_linear_solve("constant", space_p=space_p, solver_parameters=sp_, print_error=True,
                                      lambda_v_bounds=(0.3924, 2.0598), lambda_p_bounds=(0.5, 2.0), **k["rhs"])
        return [("stationary_stokes", c)]

    def stationary_navier_stokes():
        q = kat.reference_navier_stokes_problem(True, nx=4)
        sq = q["sq"]
        v_d, v_hat = q["v_d"][0], q["v_hat"][0]
        c = Control.Stationary(q["M"], lambda v, gn: q["D_v"](v, 0.0), desired_state=lambda: (v_d, v_hat),
                               beta=q["beta"], bc_dofs=q["bdofs"], bc_values=q["bc_values"][-1])
        space_p = dict(B=q["B"], M_p=sq["M_p"], K_p=sq["L_p"], forward_matrix_p=lambda v, gn: q["D_p"](v, 0.0))
        c.incompressible_non_linear_solve("constant", space_p=space_p, solver_parameters=dict(SP, relative_tolerance=1e-9),
                                          lambda_v_bounds=q["lambda_v_bounds"], lambda_p_bounds=q["lambda_p_bounds"],
                                          print_error_linear=True, print_error_non_linear=True)
        return [("stationary_navier_stokes", c)]

    def heat_inhomogeneous(CN, gn):
        nx, n_t = 6, 5
        q = kat.heat_problem(nx, n_t, CN, beta=1e-2)
        Dv = fem.nonlinear_diffusion_p1_2d(nx, nx, 2.0, 2.0)
        xb, yb = q["coords"][q["bdofs"], 0], q["coords"][q["bdofs"], 1]
        g = 0.3 * np.stack([np.cos(xb + t) + 0.5 * yb for t in q["tau"] * np.arange(n_t)])
        lv = _level(q["tau"])
        c = Control.Instationary(q["M"], lambda v, t, gn_: Dv(v, gn_),
                                 desired_state=lambda t: (q["v_d"][lv(t)], q["v_hat"][lv(t)]),
                                 force_f=lambda t: q["f"][lv(t)], beta=q["beta"], Gauss_Newton=gn, n_t=n_t, CN=CN,
                                 time_interval=q["time_interval"], bc_dofs=q["bdofs"], bc_values=lambda t: g[lv(t)])
        c.non_linear_solve(lambda_v_bounds=q["lambda_v_bounds"], solver_parameters=SP, max_non_linear_iter=6,
                           print_error_linear=True, print_error_non_linear=True)
        return [(f"heat_non_linear_cn{int(CN)}_gn{int(gn)}", c)]

    yield "stationary_heat", stationary_heat
    for CN in (True, False):
        yield f"convection_diffusion_cn{int(CN)}", lambda CN=CN: convection_diffusion(CN)
    for CN in (True, False):
        yield f"navier_stokes_cn{int(CN)}", lambda CN=CN: navier_stokes(CN)
    yield "stationary_stokes", stationary_stokes
    yield "stationary_navier_stokes", stationary_navier_stokes
    for CN, gn in ((True, False), (False, False), (True, True)):
        yield f"heat_non_linear_cn{int(CN)}_gn{int(gn)}", lambda CN=CN, gn=gn: heat_inhomogeneous(CN, gn)


def dump(out):
    Control = _stand_ins()
    arrays, text = {}, []
    for name, run in scenarios(Control):
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            results = run()
        text.append(f"=== {name}\n{buf.getvalue()}")
        for key, c in results:
            for field in FIELDS:
                if hasattr(c, field):
                    arrays[f"{key}/{field}"] = np.asarray(getattr(c, field))
    np.savez(out + ".npz", **arrays)
    with open(out + ".txt", "w") as fh:
        fh.write("".join(text))
    print(f"{len(arrays)} arrays -> {out}.npz, {sum(t.count(chr(10)) for t in text)} lines -> {out}.txt")


def compare(a, b):
    A, B = np.load(a + ".npz"), np.load(b + ".npz")
    bad = sorted(set(A.files) ^ set(B.files))
    bad += [k for k in sorted(set(A.files) & set(B.files))
            if A[k].dtype != B[k].dtype or A[k].shape != B[k].shape or A[k].tobytes() != B[k].tobytes()]
    ta, tb = open(a + ".txt").read().splitlines(), open(b + ".txt").read().splitlines()
    print(f"{len(A.files)} / {len(B.files)} arrays, differing or missing: {bad or 'none'}")
    print(f"{len(ta)} / {len(tb)} output lines, identical: {ta == tb}")
    return not bad and ta == tb


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("out", nargs="?", help="output prefix (writes <out>.npz and <out>.txt)")
    ap.add_argument("--compare", nargs=2, metavar=("A", "B"), help="compare two output prefixes")
    args = ap.parse_args()
    if args.compare:
        sys.exit(0 if compare(*args.compare) else 1)
    if not args.out:
        ap.error("give an output prefix or --compare A B")
    dump(args.out)
