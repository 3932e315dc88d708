"""Stokes control on several ranks: the two rectangular exchange plans of the divergence products (host logic,
world_size-2 gloo on CPU), the argument checks of the Python layer, and -- when at least two GPUs are present -- the
NCCL path of the CUDA library against the single-rank oracle (tests/mp_stokes_check.py under torchrun)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from control_b200 import partition
from synthetic import problems

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _B(nx=5):
    B = problems.stokes_problem(nx, 3)["th"]["B"].tocsr()
    B.sort_indices()
    return B


def _plans(A, world):
    return [partition.halo_plan(A.indptr, A.indices, world, r, n_cols=A.shape[1]) for r in range(world)]


@pytest.mark.parametrize("world", [2, 3, 4])
def test_rectangular_plans_are_consistent_between_ranks(world):
    B = _B()
    n_p, n_v = B.shape
    for A in (B, B.T.tocsr()):
        n_rows, n_cols = A.shape
        plans = _plans(A, world)
        for r, pr in enumerate(plans):
            assert (pr["row_begin"], pr["n_local"]) == partition.ownership_range(n_rows, world, r)
            assert (pr["col_begin"], pr["n_col_local"]) == partition.ownership_range(n_cols, world, r)
            # the ghosts are exactly the foreign columns this rank's rows read
            cols = np.unique(A.indices[A.indptr[pr["row_begin"]]:A.indptr[pr["row_begin"] + pr["n_local"]]])
            own = (cols >= pr["col_begin"]) & (cols < pr["col_begin"] + pr["n_col_local"])
            assert np.array_equal(pr["ghosts"], cols[~own])
            covered = 0
            for p, (off, cnt) in pr["recv"].items():
                wanted = pr["ghosts"][off:off + cnt]
                sent = plans[p]["send"][r] + plans[p]["col_begin"]
                assert np.array_equal(wanted, sent)      # same rows, same order, no negotiation
                covered += cnt
            assert covered == pr["ghosts"].size
        assert sum(p["ghosts"].size for p in plans) > 0  # the partition does cut B at this size


def test_square_plan_is_unchanged_by_the_column_split():
    """The mesh plan of the heat path is the square case of the rectangular one."""
    A = problems.heat_problem(8, 3)["M"].tocsr()
    for world in (2, 3):
        for r in range(world):
            a = partition.halo_plan(A.indptr, A.indices, world, r)
            b = partition.halo_plan(A.indptr, A.indices, world, r, n_cols=A.shape[0])
            assert np.array_equal(a["ghosts"], b["ghosts"]) and a["recv"] == b["recv"]
            assert all(np.array_equal(a["send"][p], b["send"][p]) for p in a["send"])


def _exchange(dist, plan, x_loc):
    """Ghost columns of x_loc (n_t, n_col_local) through the plan, as comm.cu::exchange_plan_run moves them."""
    ghost = np.zeros((x_loc.shape[0], plan["ghosts"].size))
    reqs, bufs = [], {}
    for p, cols in plan["send"].items():
        reqs.append(dist.isend(torch.from_numpy(np.ascontiguousarray(x_loc[:, cols])), p))
    for p, (off, cnt) in plan["recv"].items():
        bufs[p] = torch.zeros((x_loc.shape[0], cnt), dtype=torch.float64)
        reqs.append(dist.irecv(bufs[p], p))
    for q in reqs:
        q.wait()
    for p, (off, cnt) in plan["recv"].items():
        ghost[:, off:off + cnt] = bufs[p].numpy()
    return ghost


def _gloo_worker(rank, world, port, n_t, out):
    import torch.distributed as dist
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    B = _B(6)
    n_p, n_v = B.shape
    tau = 0.25
    rng = np.random.default_rng(0)
    X_v = rng.standard_normal((n_t, n_v))                # global, same on every rank
    X_p = rng.standard_normal((n_t, n_p))
    err = 0.0
    for A, X in ((B, X_v), (B.T.tocsr(), X_p)):
        plan = partition.halo_plan(A.indptr, A.indices, world, rank, n_cols=A.shape[1])
        x_loc = partition.local_blocks(X, A.shape[1], world, rank)
        ghost = _exchange(dist, plan, x_loc)
        y_loc = tau * (partition.local_rows(A, plan) @ np.concatenate([x_loc, ghost], axis=1).T).T
        y_ref = partition.local_blocks(tau * (A @ X.T).T, A.shape[0], world, rank)
        err = max(err, np.abs(y_loc - y_ref).max() / np.abs(y_ref).max())
    out[rank] = float(err)
    dist.destroy_process_group()


def test_partitioned_divergence_products_with_gloo_world_size_2():
    import torch.multiprocessing as mp
    world = 2
    with mp.Manager() as m:
        out = m.dict()
        port = 31500 + (os.getpid() % 2000)
        mp.spawn(_gloo_worker, args=(world, port, 5, out), nprocs=world, join=True)
        assert all(out[r] < 1e-13 for r in range(world)), dict(out)


# ---------------------------------------------------------------- argument checks (no device work)
def _control(world, **kw):
    from control_b200 import Control
    q = problems.stokes_problem(3, 3)
    th = q["th"]
    c = Control.Instationary(q["M"], q["K"], n_t=3, beta=1.0, CN=True, bc_dofs=q["bdofs"], rank=0, world=world, **kw)
    c.set_space_p(dict(B=th["B"], M_p=th["M_p"], K_p=th["K_p"]))
    return c


def test_several_ranks_refuse_the_one_rank_paths():
    c = _control(2)
    with pytest.raises(ValueError, match="one rank"):
        c.incompressible_linear_solve(P=lambda u0, u1, b0, b1: None)
    with pytest.raises(ValueError, match="one rank"):
        c.incompressible_non_linear_solve(device_loop=True)
    with pytest.raises(ValueError, match="one rank"):
        c.incompressible_non_linear_solve(P=lambda u0, u1, b0, b1: None)
    with pytest.raises(ValueError, match="world > 1"):
        _control(2, block_size=2)


def test_stokes_system_refuses_block_scalar_sweeps_on_several_ranks():
    from control_b200.stokes import StokesSystem
    th = problems.stokes_problem(3, 3)["th"]
    with pytest.raises(ValueError, match="world > 1"):
        StokesSystem(th["M_v"], th["K_v"], th["B"], th["M_p"], th["K_p"], n_t=3, beta=1.0, CN=True,
                     bc_dofs_v=th["bdofs_v"], velocity_block_size=2, rank=1, world=2)


# ---------------------------------------------------------------- the library on several GPUs
def _run_mp(world):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(29700 + os.getpid() % 1000),
           os.path.join(ROOT, "tests", "mp_stokes_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=1800)
    assert "MP_STOKES_CHECK_OK" in res.stdout, res.stdout[-4000:] + res.stderr[-4000:]


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4])
def test_multi_gpu_stokes_matches_oracle(world):
    """2 ranks: each has one neighbour; 4 ranks: the middle ranks exchange with peers on both sides."""
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs at least {world} GPUs")
    _run_mp(world)
