// Smoothed-aggregation AMG setup on the host, once per distinct matrix (the reference
// re-runs BoomerAMG setup 2N times per preconditioner application:
// control/control.py:2056-2067, 2098-2109, 2139-2150, 2172-2183).
#include "amg_setup.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <stdexcept>

#include <thread>

namespace {
// Rows [0, n) in contiguous blocks on up to `threads` host threads; fn(block, begin, end).  Every row is
// computed exactly as in the sequential code, so results do not depend on the thread count.
template <typename F>
void parallel_row_blocks(int n, int threads, F fn)
{
    const int T = (n < 20000 || threads <= 1) ? 1 : threads;
    if (T == 1) {
        fn(0, 0, n);
        return;
    }
    std::vector<std::thread> pool;
    for (int t = 0; t < T; ++t) {
        const int b = (int)((int64_t)n * t / T), e = (int)((int64_t)n * (t + 1) / T);
        pool.emplace_back([=, &fn]() { fn(t, b, e); });
    }
    for (auto &th : pool) th.join();
}

int row_block_count(int n, int threads) { return (n < 20000 || threads <= 1) ? 1 : threads; }

// CTL_SETUP_TIMING=1: phase times of the host setup on stderr
struct PhaseTimer {
    bool on;
    std::chrono::steady_clock::time_point t;
    PhaseTimer() : on(getenv("CTL_SETUP_TIMING") != nullptr), t(std::chrono::steady_clock::now()) {}
    void lap(const char *what, int level)
    {
        if (!on) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[ctl setup] level %d %-12s %.3f s\n", level, what, std::chrono::duration<double>(now - t).count());
        t = now;
    }
};
}  // namespace

void csr_transpose(const HostCSR &A, HostCSR &At)
{
    At.n_rows = A.n_cols;
    At.n_cols = A.n_rows;
    At.indptr.assign(A.n_cols + 1, 0);
    At.indices.resize(A.indices.size());
    At.values.resize(A.values.size());
    for (int c : A.indices) At.indptr[c + 1]++;
    for (int i = 0; i < A.n_cols; ++i) At.indptr[i + 1] += At.indptr[i];
    std::vector<int> pos(At.indptr.begin(), At.indptr.end() - 1);
    for (int r = 0; r < A.n_rows; ++r)
        for (int k = A.indptr[r]; k < A.indptr[r + 1]; ++k) {
            const int q = pos[A.indices[k]]++;
            At.indices[q] = r;
            At.values[q] = A.values[k];
        }
}

// Gustavson SpGEMM; accumulation order = ascending k of A's row, then B's row order
// (the order scipy's csr_matmat uses), columns of C sorted.
void csr_matmat(const HostCSR &A, const HostCSR &B, HostCSR &C, int threads)
{
    C.n_rows = A.n_rows;
    C.n_cols = B.n_cols;
    C.indptr.assign(A.n_rows + 1, 0);
    const int T = row_block_count(A.n_rows, threads);
    std::vector<std::vector<int>> bi(T);
    std::vector<std::vector<double>> bv(T);
    parallel_row_blocks(A.n_rows, threads, [&](int t, int r0, int r1) {
        std::vector<double> acc(B.n_cols, 0.0);
        std::vector<int> mark(B.n_cols, -1), cols;
        std::vector<int> &oi = bi[t];
        std::vector<double> &ov = bv[t];
        oi.reserve((size_t)(A.indptr[r1] - A.indptr[r0]) * 2);      // fewer regrowths (and their page faults)
        ov.reserve((size_t)(A.indptr[r1] - A.indptr[r0]) * 2);
        for (int i = r0; i < r1; ++i) {
            cols.clear();
            for (int k = A.indptr[i]; k < A.indptr[i + 1]; ++k) {
                const int j = A.indices[k];
                const double a = A.values[k];
                for (int q = B.indptr[j]; q < B.indptr[j + 1]; ++q) {
                    const int c = B.indices[q];
                    if (mark[c] != i) {
                        mark[c] = i;
                        acc[c] = 0.0;
                        cols.push_back(c);
                    }
                    acc[c] += a * B.values[q];
                }
            }
            std::sort(cols.begin(), cols.end());
            for (int c : cols) {
                oi.push_back(c);
                ov.push_back(acc[c]);
            }
            C.indptr[i + 1] = (int)cols.size();
        }
    });
    for (int i = 0; i < A.n_rows; ++i) C.indptr[i + 1] += C.indptr[i];
    C.indices.resize(C.indptr[A.n_rows]);
    C.values.resize(C.indptr[A.n_rows]);
    parallel_row_blocks(A.n_rows, threads, [&](int t, int r0, int) {
        std::copy(bi[t].begin(), bi[t].end(), C.indices.begin() + C.indptr[r0]);
        std::copy(bv[t].begin(), bv[t].end(), C.values.begin() + C.indptr[r0]);
    });
}

// oracle/amg.py:_aggregate
static int aggregate(const HostCSR &A, double theta, std::vector<int> &agg)
{
    const int n = A.n_rows;
    std::vector<double> diag(n, 0.0);
    for (int i = 0; i < n; ++i)
        for (int k = A.indptr[i]; k < A.indptr[i + 1]; ++k)
            if (A.indices[k] == i) diag[i] = A.values[k];
    std::vector<char> strong(A.indices.size(), 0);
    const double th2 = theta * theta;
    for (int i = 0; i < n; ++i)
        for (int k = A.indptr[i]; k < A.indptr[i + 1]; ++k) {
            const int j = A.indices[k];
            if (j != i) {
                const double a = A.values[k];
                if (a != 0.0 && a * a >= th2 * std::fabs(diag[i] * diag[j])) strong[k] = 1;
            }
        }
    agg.assign(n, -1);
    int n_agg = 0;
    for (int i = 0; i < n; ++i) {                       // pass 1
        if (agg[i] != -1) continue;
        bool has_nbr = false, free_ = true;
        for (int k = A.indptr[i]; k < A.indptr[i + 1]; ++k)
            if (strong[k]) {
                has_nbr = true;
                if (agg[A.indices[k]] != -1) {
                    free_ = false;
                    break;
                }
            }
        if (has_nbr && free_) {
            agg[i] = n_agg;
            for (int k = A.indptr[i]; k < A.indptr[i + 1]; ++k)
                if (strong[k]) agg[A.indices[k]] = n_agg;
            ++n_agg;
        }
    }
    const std::vector<int> agg1 = agg;                  // pass 2
    for (int i = 0; i < n; ++i) {
        if (agg1[i] != -1) continue;
        int best = -1;
        double best_val = -1.0;
        for (int k = A.indptr[i]; k < A.indptr[i + 1]; ++k)
            if (strong[k] && agg1[A.indices[k]] != -1) {
                const double a = std::fabs(A.values[k]);
                if (a > best_val) {
                    best_val = a;
                    best = agg1[A.indices[k]];
                }
            }
        if (best != -1) agg[i] = best;
    }
    for (int i = 0; i < n; ++i) {                       // pass 3
        if (agg[i] != -1) continue;
        bool has_nbr = false;
        for (int k = A.indptr[i]; k < A.indptr[i + 1]; ++k)
            if (strong[k]) {
                has_nbr = true;
                break;
            }
        if (!has_nbr) continue;
        agg[i] = n_agg;
        for (int k = A.indptr[i]; k < A.indptr[i + 1]; ++k)
            if (strong[k] && agg[A.indices[k]] == -1) agg[A.indices[k]] = n_agg;
        ++n_agg;
    }
    return n_agg;
}

static double gershgorin_rho(const HostCSR &A, std::vector<double> &dinv)
{
    const int n = A.n_rows;
    dinv.assign(n, 0.0);
    double rho = 0.0;
    for (int i = 0; i < n; ++i) {
        double d = 0.0, s = 0.0;
        for (int k = A.indptr[i]; k < A.indptr[i + 1]; ++k) {
            s += std::fabs(A.values[k]);
            if (A.indices[k] == i) d = A.values[k];
        }
        if (d == 0.0) throw std::runtime_error("AMG setup: zero diagonal entry");
        dinv[i] = 1.0 / d;
        rho = std::max(rho, s / std::fabs(d));
    }
    return rho;
}

// POWER_ITS steps of the power method on D^-1 A from a fixed start vector (oracle/amg.py::power_rho):
// a lower estimate of lambda_max(D^-1 A)
constexpr int POWER_ITS = 30;
constexpr double POWER_SAFETY = 1.2;

// stop_at > 0: the caller only needs min(stop_at, POWER_SAFETY * estimate), so the iteration ends as soon
// as the estimate is large enough for the minimum to be stop_at (the fine-mesh matrix, whose Gershgorin
// bound is sharp, leaves after a few steps instead of 30 products with 7 M entries)
static double power_rho(const HostCSR &A, const std::vector<double> &dinv, double stop_at, int threads)
{
    const int n = A.n_rows;
    std::vector<double> x(n), y(n);
    for (int i = 0; i < n; ++i) x[i] = std::sin(0.37 * (double)i + 0.1) + 0.5 * std::cos(1.3 * (double)i);
    double lam = 0.0;
    for (int it = 0; it < POWER_ITS; ++it) {
        parallel_row_blocks(n, threads, [&](int, int r0, int r1) {
            for (int i = r0; i < r1; ++i) {
                double s = 0.0;
                for (int k = A.indptr[i]; k < A.indptr[i + 1]; ++k) s += A.values[k] * x[A.indices[k]];
                y[i] = dinv[i] * s;
            }
        });
        double yy = 0.0, xx = 0.0;               // sequential sums: the result must not depend on the thread count
        for (int i = 0; i < n; ++i) {
            yy += y[i] * y[i];
            xx += x[i] * x[i];
        }
        const double ny = std::sqrt(yy);
        if (ny == 0.0) return 0.0;
        lam = ny / std::sqrt(xx);
        if (stop_at > 0.0 && POWER_SAFETY * lam >= stop_at) return lam;
        for (int i = 0; i < n; ++i) x[i] = y[i] / ny;
    }
    return lam;
}

// Gauss-Jordan with partial pivoting on [A + shift shift^T | I]; A is small (coarsest level).
// shift empty: plain inverse.  shift = normalised kernel vector e of a singular symmetric A:
// the result minus e e^T is the pseudo-inverse.
static void dense_inverse(const HostCSR &A, const std::vector<double> &shift, std::vector<double> &inv)
{
    const int n = A.n_rows;
    std::vector<double> a((size_t)n * n, 0.0);
    inv.assign((size_t)n * n, 0.0);
    for (int i = 0; i < n; ++i) {
        inv[(size_t)i * n + i] = 1.0;
        for (int k = A.indptr[i]; k < A.indptr[i + 1]; ++k) a[(size_t)i * n + A.indices[k]] += A.values[k];
    }
    if (!shift.empty())
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) a[(size_t)i * n + j] += shift[i] * shift[j];
    for (int c = 0; c < n; ++c) {
        int piv = c;
        for (int r = c + 1; r < n; ++r)
            if (std::fabs(a[(size_t)r * n + c]) > std::fabs(a[(size_t)piv * n + c])) piv = r;
        if (a[(size_t)piv * n + c] == 0.0) throw std::runtime_error("AMG setup: singular coarse matrix");
        if (piv != c)
            for (int j = 0; j < n; ++j) {
                std::swap(a[(size_t)piv * n + j], a[(size_t)c * n + j]);
                std::swap(inv[(size_t)piv * n + j], inv[(size_t)c * n + j]);
            }
        const double d = 1.0 / a[(size_t)c * n + c];
        // columns < c of the pivot row are already eliminated (exact zeros): skipping them changes nothing
        for (int j = c; j < n; ++j) a[(size_t)c * n + j] *= d;
        for (int j = 0; j < n; ++j) inv[(size_t)c * n + j] *= d;
        for (int r = 0; r < n; ++r) {
            if (r == c) continue;
            const double f = a[(size_t)r * n + c];
            if (f == 0.0) continue;
            const double *ac = &a[(size_t)c * n], *ic = &inv[(size_t)c * n];
            double *ar = &a[(size_t)r * n], *ir = &inv[(size_t)r * n];
            for (int j = c; j < n; ++j) ar[j] -= f * ac[j];
            for (int j = 0; j < n; ++j) ir[j] -= f * ic[j];
        }
    }
}

int setup_threads(int fallback)
{
    if (const char *e = getenv("CTL_SETUP_THREADS")) return atoi(e);
    return fallback;
}

void amg_setup_host(const HostCSR &A0, const AmgParams &p, std::vector<AmgLevelHost> &levels, int threads)
{
    if (threads <= 0) threads = std::max(1, std::min(setup_threads((int)std::thread::hardware_concurrency()), 32));
    levels.clear();
    levels.reserve((size_t)std::max(1, p.max_levels));      // references to a level stay valid while the next is built
    HostCSR next = A0;                                       // the one copy: the caller keeps its matrix
    std::vector<double> cand(A0.n_rows, 1.0);
    PhaseTimer timer;
    while (true) {
        levels.emplace_back();
        AmgLevelHost &L = levels.back();
        const int lvl = (int)levels.size() - 1;
        L.A = std::move(next);
        const HostCSR &A = L.A;
        timer.lap("copy", lvl);
        L.rho = gershgorin_rho(L.A, L.dinv);
        L.rho = std::min(L.rho, POWER_SAFETY * power_rho(L.A, L.dinv, L.rho, threads));
        timer.lap("rho", lvl);
        const int n = A.n_rows;
        if (n <= p.coarse_max || (int)levels.size() >= p.max_levels) break;
        std::vector<int> agg;
        const int n_agg = aggregate(A, p.theta * std::pow(p.theta_decay, (double)(levels.size() - 1)), agg);
        if (n_agg == 0 || n_agg >= 0.9 * n) break;
        L.agg = agg;
        timer.lap("aggregate", lvl);
        // tentative prolongator from the near-kernel candidate: T_jJ = cand_j / ||cand|agg_J||,
        // coarse candidate = those norms
        std::vector<double> norms(n_agg, 0.0), t(n, 0.0);
        for (int i = 0; i < n; ++i)
            if (agg[i] >= 0) norms[agg[i]] += cand[i] * cand[i];
        for (int J = 0; J < n_agg; ++J) norms[J] = std::sqrt(norms[J]);
        for (int i = 0; i < n; ++i)
            if (agg[i] >= 0) t[i] = cand[i] / norms[agg[i]];
        // P = T - diag(omega * dinv) (A T), explicit zeros of A skipped
        const double omega = 4.0 / (3.0 * L.rho);
        HostCSR &P = L.P;
        P.n_rows = n;
        P.n_cols = n_agg;
        P.indptr.assign(n + 1, 0);
        {
            const int T = row_block_count(n, threads);
            std::vector<std::vector<int>> bi(T);
            std::vector<std::vector<double>> bv(T);
            parallel_row_blocks(n, threads, [&](int tb, int r0, int r1) {
                std::vector<std::pair<int, double>> row;
                for (int i = r0; i < r1; ++i) {
                    row.clear();
                    // (A T)_iJ accumulated in CSR order of j
                    for (int k = A.indptr[i]; k < A.indptr[i + 1]; ++k) {
                        const double a = A.values[k];
                        const int j = A.indices[k], J = agg[j];
                        if (a == 0.0 || J < 0) continue;
                        auto it = std::find_if(row.begin(), row.end(), [J](const std::pair<int, double> &e) { return e.first == J; });
                        if (it == row.end()) row.emplace_back(J, a * t[j]);
                        else it->second += a * t[j];
                    }
                    const double d = omega * L.dinv[i];
                    for (auto &e : row) e.second = -(d * e.second);
                    if (agg[i] >= 0) {
                        const int J = agg[i];
                        auto it = std::find_if(row.begin(), row.end(), [J](const std::pair<int, double> &e) { return e.first == J; });
                        if (it == row.end()) row.emplace_back(J, t[i]);
                        else it->second = t[i] + it->second;
                    }
                    std::sort(row.begin(), row.end());
                    for (auto &e : row) {
                        bi[tb].push_back(e.first);
                        bv[tb].push_back(e.second);
                    }
                    P.indptr[i + 1] = (int)row.size();
                }
            });
            for (int i = 0; i < n; ++i) P.indptr[i + 1] += P.indptr[i];
            P.indices.resize(P.indptr[n]);
            P.values.resize(P.indptr[n]);
            parallel_row_blocks(n, threads, [&](int tb, int r0, int) {
                std::copy(bi[tb].begin(), bi[tb].end(), P.indices.begin() + P.indptr[r0]);
                std::copy(bv[tb].begin(), bv[tb].end(), P.values.begin() + P.indptr[r0]);
            });
        }
        timer.lap("prolongator", lvl);
        csr_transpose(P, L.R);
        timer.lap("transpose", lvl);
        HostCSR AP, Ac;
        csr_matmat(A, P, AP, threads);
        timer.lap("A*P", lvl);
        csr_matmat(L.R, AP, Ac, threads);
        timer.lap("R*(AP)", lvl);
        next = std::move(Ac);
        cand = norms;
    }
    AmgLevelHost &last = levels.back();
    if (last.A.n_rows <= 4096 && p.coarse == AMG_COARSE_INVERSE) {
        if (p.device_inverse) last.coarse_inverse = AMG_COARSE_INVERSE + 1;
        else dense_inverse(last.A, {}, last.Ainv);
    } else if (last.A.n_rows <= 4096 && p.coarse == AMG_COARSE_PINV_CONSTANT) {
        // kernel of the coarsest Galerkin operator = the coarse image of the constants
        const int nc = last.A.n_rows;
        double nn = 0.0;
        for (double c : cand) nn += c * c;
        nn = std::sqrt(nn);
        std::vector<double> e(nc);
        for (int i = 0; i < nc; ++i) e[i] = cand[i] / nn;
        if (p.device_inverse) {
            last.coarse_inverse = AMG_COARSE_PINV_CONSTANT + 1;
            last.coarse_shift = e;
        } else {
            dense_inverse(last.A, e, last.Ainv);
            for (int i = 0; i < nc; ++i)
                for (int j = 0; j < nc; ++j) last.Ainv[(size_t)i * nc + j] -= e[i] * e[j];
        }
    }
    timer.lap("coarse solve", (int)levels.size() - 1);
}
