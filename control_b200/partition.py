"""Row partition of the spatial dofs over ranks (host-side mirror of the plan the CUDA
library derives in csrc/api.cu + csrc/comm.cu).

The reference distributes its matrices and vectors the PETSc way: every rank owns a
contiguous block of rows of every time block (preconditioner/preconditioner.py:706-722 sizes
the shell matrix ((n_local, N_global), ...)).  ``ownership_range`` is PETSc's
``PetscSplitOwnership`` rule; ``halo_plan`` lists, for one rank, the ghost columns it reads
(sorted by global index = grouped by owner) and the owned rows every peer reads from it.
No communication is needed to build the plan: every rank holds the global pattern.  The rows and
the columns may belong to two spaces, each split on its own (``n_cols``): the divergence matrix
``B`` of the Stokes system (pressure rows, velocity columns) and its transpose
(csrc/comm.cu::exchange_plan_build, csrc/stokes.cu).
"""
import numpy as np

__all__ = ["ownership_range", "halo_plan", "local_rows", "local_blocks", "gather_blocks"]


def ownership_range(n, world, rank):
    """(first owned row, number of owned rows)."""
    base, rem = divmod(n, world)
    return rank * base + min(rank, rem), base + (1 if rank < rem else 0)


def halo_plan(indptr, indices, world, rank, n_cols=None):
    """dict(ghosts=global ids of this rank's ghost columns (sorted),
            recv={peer: (offset into ghosts, count)},
            send={peer: local owned columns the peer needs, in the peer's ghost order},
            row_begin / n_local: this rank's rows, col_begin / n_col_local: its columns).
    ``n_cols``: columns of a rectangular pattern, split on their own (default: square)."""
    n = len(indptr) - 1
    n_cols = n if n_cols is None else int(n_cols)
    rb, nl = ownership_range(n, world, rank)
    cb, nc = ownership_range(n_cols, world, rank)
    cols = np.unique(indices[indptr[rb]:indptr[rb + nl]])
    ghosts = cols[(cols < cb) | (cols >= cb + nc)]
    recv, send = {}, {}
    for p in range(world):
        if p == rank:
            continue
        pr, prc = ownership_range(n, world, p)
        pb, pc = ownership_range(n_cols, world, p)
        lo, hi = np.searchsorted(ghosts, [pb, pb + pc])
        pcols = np.unique(indices[indptr[pr]:indptr[pr + prc]])
        need = pcols[(pcols >= cb) & (pcols < cb + nc)]
        if hi > lo or need.size:
            recv[p] = (int(lo), int(hi - lo))
            send[p] = (need - cb).astype(np.int64)
    return dict(ghosts=ghosts.astype(np.int64), recv=recv, send=send, row_begin=rb, n_local=nl, col_begin=cb,
                n_col_local=nc)


def local_rows(A, plan):
    """This rank's rows of the global CSR ``A`` in the plan's local column numbering: owned columns first, then the
    ghosts (csrc/stokes.cu::local_rows).  Entries keep their order within a row."""
    import scipy.sparse as sp
    A = A.tocsr()
    rb, nl, cb, nc = plan["row_begin"], plan["n_local"], plan["col_begin"], plan["n_col_local"]
    ghosts = plan["ghosts"]
    rows = A[rb:rb + nl]
    own = (rows.indices >= cb) & (rows.indices < cb + nc)
    idx = np.where(own, rows.indices - cb, nc + np.searchsorted(ghosts, rows.indices))
    return sp.csr_matrix((rows.data, idx, rows.indptr), shape=(nl, nc + ghosts.size))


def local_blocks(x, n, world, rank):
    """This rank's columns of a global block array (N, n)."""
    rb, nl = ownership_range(n, world, rank)
    return np.ascontiguousarray(np.asarray(x)[:, rb:rb + nl])


def gather_blocks(parts):
    """Inverse of ``local_blocks`` over all ranks (list ordered by rank)."""
    return np.concatenate(parts, axis=1)
