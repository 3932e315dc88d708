"""Host logic of bench.py without a GPU: option parsing, the committed one-GPU records the multi-GPU lines and the CPU
arm refer to, and the JSON contract of the reference arm on a small problem."""
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def _args(**kw):
    d = dict(workload="heat", nx=1024, n_t=64, ksp="minres", rtol=1e-6, amg="cycles=2,nu=4", ref_its=None, gpus=1)
    d.update(kw)
    return types.SimpleNamespace(**d)


def test_amg_options_and_keys():
    assert bench.amg_options("cycles=2,nu=4") == {"cycles": 2, "nu": 4}
    assert bench.amg_options("") == {} and bench.amg_options(None) == {}
    assert bench.amg_options("lo=0.3,cycles=3") == {"lo": 0.3, "cycles": 3}
    assert bench.problem_key(_args()) == "heat/1024/64/minres/1e-06/cycles=2,nu=4"
    assert bench.problem_key(_args(workload="c3", nx=128, n_t=32, ksp="gmres", amg="")) == "c3/128/32/gmres/1e-06"


def test_one_gpu_records_cover_the_bench_configurations():
    """Every configuration bench.py runs by default has a committed one-GPU record (iterations, true residual)."""
    for a in (_args(), _args(ksp="fgmres", amg=""), _args(workload="c3", nx=128, n_t=32, ksp="gmres", amg="")):
        rec = bench.n1_expectation(a)
        assert rec is not None and rec["iterations"] > 0 and rec["kkt_residual"] > 0.0, bench.problem_key(a)
        its, source = bench.known_iterations(a)
        assert its == rec["iterations"] and "iteration_counts.json" in source
    assert bench.known_iterations(_args(ref_its=7)) == (7, "--ref_its")
    assert bench.known_iterations(_args(nx=999))[1].startswith("assumed")


def test_dump_sample_is_the_same_for_any_row_partition(tmp_path, monkeypatch):
    """--dump-outputs: the sample is drawn in global (block, dof) numbering, so one rank and a row partition over two
    ranks dump the same entries; small blocks are written whole."""
    import numpy as np
    import torch
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 50)
    N, n = 7, 13
    rng = np.random.default_rng(3)
    v, zeta = rng.standard_normal((N, n)), rng.standard_normal((N, n))
    whole = bench.sample_blocks(torch.from_numpy(np.concatenate([v.ravel(), zeta.ravel()])),
                                [("v", 0, N, n, 0, n), ("zeta", N * n, N, n, 0, n)])
    assert 0 < whole["v"].size <= 50 and np.all(np.isin(whole["v"], v)) and np.all(np.isin(whole["zeta"], zeta))
    split = {"v": 0.0, "zeta": 0.0}
    for rb, nl in ((0, 7), (7, 6)):                    # two ranks; their sum plays the all-reduce
        u = torch.from_numpy(np.concatenate([v[:, rb:rb + nl].ravel(), zeta[:, rb:rb + nl].ravel()]))
        part = bench.sample_blocks(u, [("v", 0, N, n, rb, nl), ("zeta", N * nl, N, n, rb, nl)])
        split = {k: split[k] + part[k] for k in split}
    assert all(np.array_equal(whole[k], split[k]) for k in split)
    small = bench.sample_blocks(torch.arange(6, dtype=torch.float64), [("p", 0, 2, 3, 0, 3)])
    assert np.array_equal(small["p"], np.arange(6.0))
    bench.write_outputs(str(tmp_path / "out"), {**whole, "residual_history": [1.0, 0.5]})
    assert sorted(os.listdir(tmp_path / "out")) == ["residual_history.npy", "v.npy", "zeta.npy"]
    assert np.load(tmp_path / "out" / "residual_history.npy").dtype == np.float64


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                         timeout=120)
    assert out.returncode == 2 and "--steps must be at least 1" in out.stderr


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm: C / OpenMP port of the reference's algorithm) on a small problem."""
    so = os.path.join(ROOT, "oracle", "_build", "liboracle.so")
    if not os.path.exists(so):
        import pytest
        pytest.skip("oracle/_build/liboracle.so not built")
    env = dict(os.environ, OMP_NUM_THREADS="1")          # what torchrun exports: the arm must override it
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--nx", "48", "--n_t", "8",
                          "--steps", "1", "--warmup", "1", "--ref_its", "5"], capture_output=True, text=True, env=env,
                         timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "kkt_solve_time" and line["unit"] == "s"
    assert line["higher_is_better"] is False and line["gpu_launches"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == line["value"] > 0.0
    assert cb["cores"] == (os.cpu_count() or 1)          # all host cores, not OMP_NUM_THREADS=1
    assert line["e2e"] == {"value": line["value"], "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["iterations"] == 5 and "2 aggregation-AMG V(4,4) cycles" in line["config"]["workload"]
