// Pure host part of the NCCL panel exchange (comm.cu) and of the local divergence matrices (stokes.cu), no CUDA
// calls: header-only so that tests/native/exchange_plan_check.cu can play all ranks of a partition in one process.
//
// A global CSR pattern whose rows and columns may belong to two spaces, each split over the ranks by PETSc's rule
// (the mesh pattern of a handle; the divergence matrix B and its transpose between the velocity and pressure
// spaces).  The rows of a rank gather its ghost columns: the columns its rows read that other ranks own.  No
// communication is needed to build the lists: every rank holds the global pattern.
#pragma once
#include <algorithm>
#include <vector>

#include "common.cuh"

// PETSc's ownership split (PetscSplitOwnership): the first n % world ranks get one extra row
inline void owner_range(int n, int world, int rank, int *begin, int *count)
{
    const int base = n / world, rem = n % world;
    *count = base + (rank < rem ? 1 : 0);
    *begin = rank * base + std::min(rank, rem);
}

struct ExchangeLists {
    std::vector<int> ghosts;              // global column of each ghost, sorted (= grouped by owner)
    std::vector<int> peers;               // ranks we exchange with
    std::vector<int> recv_off, recv_cnt;  // ghost segment of each peer (rows)
    std::vector<int> send_off, send_cnt;  // segment of each peer in send_rows
    std::vector<int> send_rows;           // owned local columns each peer reads, peer after peer, in its ghost order
};

// the lists of rank `me` for the rows [row split of n_rows] over the columns [column split of n_cols]
inline void exchange_lists(const int *ip, const int *ix, int n_rows, int n_cols, int world, int me, ExchangeLists &P)
{
    int my_r, my_rc, my_b, my_c;
    owner_range(n_rows, world, me, &my_r, &my_rc);
    owner_range(n_cols, world, me, &my_b, &my_c);
    P = ExchangeLists();
    std::vector<int> &ghosts = P.ghosts;
    for (int r = my_r; r < my_r + my_rc; ++r)
        for (int k = ip[r]; k < ip[r + 1]; ++k)
            if (ix[k] < my_b || ix[k] >= my_b + my_c) ghosts.push_back(ix[k]);
    std::sort(ghosts.begin(), ghosts.end());
    ghosts.erase(std::unique(ghosts.begin(), ghosts.end()), ghosts.end());
    for (int p = 0; p < world; ++p) {
        if (p == me) continue;
        int pr, prc, pb, pc;
        owner_range(n_rows, world, p, &pr, &prc);
        owner_range(n_cols, world, p, &pb, &pc);
        // what p needs from me: columns in my range referenced by p's rows (sorted, unique):
        // exactly the segment of p's ghost list that I own, in p's ghost order
        std::vector<int> need;
        for (int r = pr; r < pr + prc; ++r)
            for (int k = ip[r]; k < ip[r + 1]; ++k)
                if (ix[k] >= my_b && ix[k] < my_b + my_c) need.push_back(ix[k]);
        std::sort(need.begin(), need.end());
        need.erase(std::unique(need.begin(), need.end()), need.end());
        // what I need from p: my ghosts in p's column range
        const auto lo = std::lower_bound(ghosts.begin(), ghosts.end(), pb);
        const auto hi = std::lower_bound(ghosts.begin(), ghosts.end(), pb + pc);
        const int rc = (int)(hi - lo);
        if (need.empty() && rc == 0) continue;
        P.peers.push_back(p);
        P.recv_off.push_back((int)(lo - ghosts.begin()));
        P.recv_cnt.push_back(rc);
        P.send_off.push_back((int)P.send_rows.size());
        P.send_cnt.push_back((int)need.size());
        for (int g : need) P.send_rows.push_back(g - my_b);
    }
}

// rows [rb, rb + nr) of a global CSR, columns renumbered: the owned range [cb, cb + nc) first, then the ghosts
// (sorted); entries keep their order within a row, so a product sums in the order of the global one
inline HostCSR local_rows(const HostCSR &A, int rb, int nr, int cb, int nc, const std::vector<int> &ghosts)
{
    HostCSR L;
    L.n_rows = nr;
    L.n_cols = nc + (int)ghosts.size();
    L.indptr.assign(1, 0);
    for (int r = rb; r < rb + nr; ++r) {
        for (int k = A.indptr[r]; k < A.indptr[r + 1]; ++k) {
            const int c = A.indices[k];
            L.indices.push_back(c >= cb && c < cb + nc
                                    ? c - cb
                                    : nc + (int)(std::lower_bound(ghosts.begin(), ghosts.end(), c) - ghosts.begin()));
            L.values.push_back(A.values[k]);
        }
        L.indptr.push_back((int)L.indices.size());
    }
    return L;
}
