// Host-only check of csrc/exchange_plan.h: plays ALL ranks of a partition in one process, for a rectangular pattern
// (rows and columns split on their own, as B and B^T between the pressure and velocity spaces), its transpose and a
// square one, at world = 2 .. 5:
//  * what each rank expects from a peer (its ghost segment) is what the peer sends it, in the same order, and the
//    segments cover every ghost;
//  * the products of the local row blocks (local_rows) with [owned rows | ghost rows delivered through the send
//    lists] equal the rows of the global product bitwise: same entries, same order.
// Built and run by tests/test_stokes_plan_native.py.
#include <cstdio>
#include <random>

#include "amg_setup.cpp"
#include "exchange_plan.h"

static int failures = 0;
#define EXPECT(c)                                                                   \
    do {                                                                            \
        if (!(c)) {                                                                 \
            ++failures;                                                             \
            std::printf("FAILED %s (line %d)\n", #c, __LINE__);                     \
        }                                                                           \
    } while (0)

// rows with a band of columns around their "position" in the column space, and one far column every 7th row
static HostCSR pattern(int n_rows, int n_cols, unsigned seed)
{
    std::mt19937 rng(seed);
    HostCSR A;
    A.n_rows = n_rows;
    A.n_cols = n_cols;
    A.indptr.assign(1, 0);
    std::uniform_real_distribution<double> val(-1.0, 1.0);
    for (int r = 0; r < n_rows; ++r) {
        std::vector<int> c;
        const int centre = (int)((long)r * n_cols / n_rows);
        for (int d = -4; d <= 4; ++d)
            if (rng() % 3 != 0) c.push_back(std::min(n_cols - 1, std::max(0, centre + d)));
        if (r % 7 == 0) c.push_back((int)(rng() % n_cols));
        std::sort(c.begin(), c.end());
        c.erase(std::unique(c.begin(), c.end()), c.end());
        for (int x : c) {
            A.indices.push_back(x);
            A.values.push_back(val(rng));
        }
        A.indptr.push_back((int)A.indices.size());
    }
    return A;
}

static void check(const HostCSR &A, int world, int ld)
{
    std::vector<ExchangeLists> L(world);
    for (int r = 0; r < world; ++r)
        exchange_lists(A.indptr.data(), A.indices.data(), A.n_rows, A.n_cols, world, r, L[r]);
    std::mt19937 rng(7);
    std::uniform_real_distribution<double> val(-1.0, 1.0);
    std::vector<double> X((size_t)A.n_cols * ld), Y((size_t)A.n_rows * ld, 0.0);      // [rows x ld] panels
    for (double &x : X) x = val(rng);
    for (int r = 0; r < A.n_rows; ++r)
        for (int k = A.indptr[r]; k < A.indptr[r + 1]; ++k)
            for (int j = 0; j < ld; ++j) Y[(size_t)r * ld + j] += A.values[k] * X[(size_t)A.indices[k] * ld + j];
    int cut = 0;
    for (int me = 0; me < world; ++me) {
        const ExchangeLists &P = L[me];
        int rb, nr, cb, nc;
        owner_range(A.n_rows, world, me, &rb, &nr);
        owner_range(A.n_cols, world, me, &cb, &nc);
        // the ghost rows as the exchange delivers them: peer after peer, out of the peer's packed send list
        std::vector<double> ghost(P.ghosts.size() * ld, -1e300);
        int covered = 0;
        for (size_t i = 0; i < P.peers.size(); ++i) {
            const int p = P.peers[i];
            const ExchangeLists &Q = L[p];
            const size_t at = std::find(Q.peers.begin(), Q.peers.end(), me) - Q.peers.begin();
            EXPECT(at < Q.peers.size());
            if (at == Q.peers.size()) continue;
            EXPECT(Q.send_cnt[at] == P.recv_cnt[i]);
            int pb, pc;
            owner_range(A.n_cols, world, p, &pb, &pc);
            for (int q = 0; q < P.recv_cnt[i] && q < Q.send_cnt[at]; ++q) {
                const int col = Q.send_rows[Q.send_off[at] + q];      // local column of p
                EXPECT(pb + col == P.ghosts[P.recv_off[i] + q]);
                for (int j = 0; j < ld; ++j) ghost[(size_t)(P.recv_off[i] + q) * ld + j] = X[(size_t)(pb + col) * ld + j];
            }
            covered += P.recv_cnt[i];
        }
        EXPECT(covered == (int)P.ghosts.size());
        cut += (int)P.ghosts.size();
        const HostCSR Ll = local_rows(A, rb, nr, cb, nc, P.ghosts);
        EXPECT(Ll.n_cols == nc + (int)P.ghosts.size());
        for (int r = 0; r < nr; ++r)
            for (int j = 0; j < ld; ++j) {
                double y = 0.0;
                for (int k = Ll.indptr[r]; k < Ll.indptr[r + 1]; ++k) {
                    const int c = Ll.indices[k];
                    const double x = c < nc ? X[(size_t)(cb + c) * ld + j] : ghost[(size_t)(c - nc) * ld + j];
                    y += Ll.values[k] * x;
                }
                EXPECT(y == Y[(size_t)(rb + r) * ld + j]);
            }
    }
    EXPECT(cut > 0);
}

int main()
{
    const HostCSR B = pattern(57, 133, 1);      // pressure rows x velocity columns
    HostCSR BT;
    csr_transpose(B, BT);
    const HostCSR S = pattern(90, 90, 2);
    for (int world = 2; world <= 5; ++world) {
        check(B, world, 4);
        check(BT, world, 4);
        check(S, world, 2);
    }
    std::printf("exchange plan check: %d failures\n", failures);
    return failures == 0 ? 0 : 1;
}
