// ============================================================================
// oracle/csw_l1.cpp — parity-ladder level L1 for the split weights (TEST INFRASTRUCTURE ONLY).
//
// Same algorithm as CircularSplitWeights.java (see nnet_oracle.cpp for the literal L0), but with
// the GPU's formulation of the two mat-vecs (2-D prefix sums + gathers) and the GPU's fixed
// reduction trees, restated on the CPU operation for operation (csrc/fnn_csw.cu).  The CUDA path
// must match THIS bit for bit; |L1 - L0| is the reference algorithm's own summation-order noise
// floor (SURVEY F5).  PARITY UNPINNED against the reference itself (no JVM, no golden vectors).
// ============================================================================
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <vector>

namespace {
inline int64_t row_start(int64_t n, int64_t i) { return i * (2 * n - i - 1) / 2; }
inline int64_t pidx(int64_t n, int64_t i, int64_t j) { return i * (2 * n - i - 3) / 2 + j - 1; }

// k_rowscan: blocks of 32, Kogge-Stone inside, carry added sequentially
void rowscan(int64_t n, const double* v, double* Rw, double* RT) {
    for (int64_t i = 0; i < n - 1; ++i) {
        const int64_t rs = row_start(n, i);
        const int len = (int)(n - 1 - i);
        double carry = 0.0;
        for (int blk = 0; blk < len; blk += 32) {
            double e[32], t[32];
            for (int l = 0; l < 32; ++l) e[l] = (blk + l < len) ? v[rs + blk + l] : 0.0;
            for (int off = 1; off < 32; off <<= 1) {
                for (int l = 0; l < 32; ++l) t[l] = (l >= off) ? e[l] + e[l - off] : e[l];
                for (int l = 0; l < 32; ++l) e[l] = t[l];
            }
            double last = 0.0;
            for (int l = 0; l < 32; ++l) {
                const double out = carry + e[l];
                if (blk + l < len) Rw[rs + blk + l] = out;
                if (l == 31) last = out;
            }
            carry = last;
        }
        if (RT) RT[i] = carry;
    }
    if (RT) RT[n - 1] = 0.0;
}
// k_colscan_local / k_colscan_carry / k_colscan_fix: chunks of 32 rows scanned from zero, sequential carry
void colscan(int64_t n, const double* Rw, const double* v, double* P, double* CT) {
    const int64_t CH = 32;
    if (CT) CT[0] = 0.0;
    for (int64_t j = 0; j < n; ++j) {
        double carry = 0.0, ct = 0.0;
        for (int64_t i0 = 0; i0 < n; i0 += CH) {   // every chunk index exists for every column (empty chunks add 0.0)
            const int64_t i1 = std::min(i0 + CH, j);
            double acc = 0.0, acc2 = 0.0;
            for (int64_t i = i0; i < i1; ++i) {
                const int64_t q = pidx(n, i, j);
                acc = acc + Rw[q];
                P[q] = carry + acc;
                if (CT) acc2 = acc2 + v[q];
            }
            carry = carry + acc;
            if (CT) ct = ct + acc2;
        }
        if (CT) CT[j] = ct;
    }
}
struct Work { std::vector<double> Rw, P, RT, CT, PRS; };

void Ab(int64_t n, const double* in, double* out, Work& w) {
    rowscan(n, in, w.Rw.data(), nullptr);
    colscan(n, w.Rw.data(), in, w.P.data(), nullptr);
    const double* P = w.P.data();
    for (int64_t a = 0; a < n - 1; ++a) {
        const double Pda = (a - 1 >= 1) ? P[pidx(n, a - 2, a - 1)] : 0.0;
        const double Prowa = (a >= 1) ? P[pidx(n, a - 1, n - 1)] : 0.0;
        for (int64_t b = a + 1; b < n; ++b) {
            const double P1 = (a >= 1) ? P[pidx(n, a - 1, b - 1)] : 0.0;
            const double Prowb = P[pidx(n, b - 1, n - 1)];
            const double Pdb = (b - 1 >= 1) ? P[pidx(n, b - 2, b - 1)] : 0.0;
            double t = 2.0 * P1;
            t = t - Pda; t = t + Prowb; t = t - Prowa; t = t - Pdb;
            out[pidx(n, a, b)] = t;
        }
    }
}
void Atx(int64_t n, const double* in, double* out, Work& w) {
    rowscan(n, in, w.Rw.data(), w.RT.data());
    colscan(n, w.Rw.data(), in, w.P.data(), w.CT.data());
    {   // prs_scan_warp: blocks of 32, Kogge-Stone inside, carry added sequentially
        double carry = 0.0;
        for (int64_t blk = 0; blk < n; blk += 32) {
            double e[32], t[32];
            for (int l = 0; l < 32; ++l) e[l] = (blk + l < n) ? w.RT[blk + l] + w.CT[blk + l] : 0.0;
            for (int off = 1; off < 32; off <<= 1) {
                for (int l = 0; l < 32; ++l) t[l] = (l >= off) ? e[l] + e[l - off] : e[l];
                for (int l = 0; l < 32; ++l) e[l] = t[l];
            }
            double last = 0.0;
            for (int l = 0; l < 32; ++l) {
                const double out = carry + e[l];
                if (blk + l < n) w.PRS[blk + l] = out;
                if (l == 31) last = out;
            }
            carry = last;
        }
    }
    const double* G = w.P.data();
    for (int64_t i = 0; i < n - 1; ++i)
        for (int64_t j = i + 1; j < n; ++j) {
            const int64_t k = pidx(n, i, j);
            const double u = w.PRS[j] - w.PRS[i];
            const double ww = G[pidx(n, j - 1, j)] - G[k];
            out[k] = u - 2.0 * ww;
        }
}
// block_tree_1024 on 1024 consecutive values (zero padded)
double block1024(const double* v, int64_t base, int64_t len) {
    double s[256];
    for (int t = 0; t < 256; ++t) {
        double e[4];
        for (int q = 0; q < 4; ++q) { const int64_t k = base + 4 * t + q; e[q] = (k < len) ? v[k] : 0.0; }
        s[t] = ((e[0] + e[1]) + e[2]) + e[3];
    }
    double wt[8];
    for (int w = 0; w < 8; ++w) {
        double x[32];
        for (int l = 0; l < 32; ++l) x[l] = s[32 * w + l];
        for (int off = 16; off > 0; off >>= 1)
            for (int l = 0; l < off; ++l) x[l] = x[l] + x[l + off];   // lane l after the xor butterfly (commutative)
        wt[w] = x[0];
    }
    double t = wt[0];
    for (int w = 1; w < 8; ++w) t = t + wt[w];
    return t;
}
double tree_sum(std::vector<double> v) {
    while (true) {
        const int64_t len = (int64_t)v.size();
        const int64_t blocks = (len + 1023) / 1024;
        std::vector<double> out(blocks);
        for (int64_t b = 0; b < blocks; ++b) out[b] = block1024(v.data(), b * 1024, len);
        if (blocks == 1) return out[0];
        v.swap(out);
    }
}
void unconstrainedLS(int64_t n, const double* d, double* x) {   // identical to L0 (no reductions)
    int64_t index = 0;
    for (int64_t i = 0; i <= n - 3; i++) {
        x[index] = (d[index] + d[index + (n - i - 2) + 1] - d[index + 1]) / 2.0; index++;
        for (int64_t j = i + 2; j <= n - 2; j++) { x[index] = (d[index] + d[index + (n - i - 2) + 1] - d[index + 1] - d[index + (n - i - 2)]) / 2.0; index++; }
        if (i == 0) x[index] = (d[0] + d[n - 2] - d[2 * n - 4]) / 2.0;
        else x[index] = (d[index] + d[i] - d[i - 1] - d[index + (n - i - 2)]) / 2.0;
        index++;
    }
    x[index] = (d[index] + d[n - 2] - d[n - 3]) / 2.0;
}
struct Stats { int64_t cg_iters = 0, cg_calls = 0, outer = 0, inner = 0; };

void conjugateGrads(int64_t n, int64_t np, std::vector<double>& r, std::vector<double>& w, std::vector<double>& p,
                    std::vector<double>& y, const std::vector<double>& b, double e0sq, const std::vector<uint8_t>& active,
                    double* x, int64_t kmax, Work& wk, Stats& st) {
    st.cg_calls++;
    Ab(n, x, y.data(), wk);
    Atx(n, y.data(), r.data(), wk);
    std::vector<double> sq(np);
    for (int64_t k = 0; k < np; ++k) { const double v = active[k] ? 0.0 : b[k] - r[k]; r[k] = v; sq[k] = v * v; }
    double rho = tree_sum(sq), rho_old = 0.0;
    int64_t k = 0;
    while ((rho > e0sq) && (k < kmax)) {
        k = k + 1;
        st.cg_iters++;
        if (k == 1) { for (int64_t i = 0; i < np; ++i) p[i] = r[i]; }
        else { const double beta = rho / rho_old; for (int64_t i = 0; i < np; ++i) p[i] = r[i] + beta * p[i]; }
        Ab(n, p.data(), y.data(), wk);
        Atx(n, y.data(), w.data(), wk);
        for (int64_t i = 0; i < np; ++i) { if (active[i]) w[i] = 0.0; sq[i] = p[i] * w[i]; }
        const double alpha = rho / tree_sum(sq);
        for (int64_t i = 0; i < np; ++i) { x[i] = x[i] + alpha * p[i]; const double rv = r[i] - alpha * w[i]; r[i] = rv; sq[i] = rv * rv; }
        rho_old = rho;
        rho = tree_sum(sq);
    }
}
// runActiveConjugate (:359-557) in the device driver's order (active_conjugate, csrc/fnn_csw.cu).  kmax: iteration cap of
// every CG call; max_cg_calls > 0: return right after that many CG calls (the budget of fnn_split_weights_budget).
void activeConjugate(int64_t n, int64_t np, const double* d, double* x, std::vector<uint8_t>& active, int64_t kmax,
                     int64_t max_cg_calls, Work& wk, Stats& st) {
    std::vector<double> r(np), w(np), p(np), y(np), old_x(np, 1.0), AtWd(np), sq(np);
    Atx(n, d, AtWd.data(), wk);
    for (int64_t k = 0; k < np; ++k) sq[k] = AtWd[k] * AtWd[k];
    const double e0 = 1e-8 * std::sqrt(tree_sum(sq));
    const double e0sq = e0 * e0;
    auto cg = [&]() {
        conjugateGrads(n, np, r, w, p, y, AtWd, e0sq, active, x, kmax, wk, st);
        return max_cg_calls > 0 && st.cg_calls >= max_cg_calls;   // budget spent
    };
    bool first_pass = true;
    while (true) {
        st.outer++;
        while (true) {
            st.inner++;
            if (!first_pass && cg()) return;
            first_pass = false;
            {   // worstIndices(x, 0.6) (CircularSplitWeights.java:282-330)
                std::vector<double> neg;
                for (int64_t i = 0; i < np; ++i) if (x[i] < 0.0) neg.push_back(x[i]);
                if (!neg.empty()) {
                    std::sort(neg.begin(), neg.end());
                    const int64_t nkept = (int64_t)std::ceil(0.6 * (double)neg.size());
                    const double cutoff = neg[nkept - 1];
                    std::vector<int64_t> result(nkept, -1);
                    int64_t front = 0, back = nkept - 1;
                    for (int64_t i = 0; i < np; ++i) {
                        if (x[i] < cutoff) result[front++] = i;
                        else if (x[i] == cutoff) { if (back >= front) result[back--] = i; }
                    }
                    for (int64_t idx : result) if (idx >= 0) { x[idx] = 0.0; active[idx] = 1; }
                    if (cg()) return;
                }
            }
            int64_t min_i = -1; double min_xi = -1.0;
            for (int64_t i = 0; i < np; ++i)
                if (x[i] < 0.0) {
                    const double xi = old_x[i] / (old_x[i] - x[i]);
                    if (min_i == -1 || xi < min_xi) { min_i = i; min_xi = xi; }
                }
            if (min_i == -1) break;
            for (int64_t i = 0; i < np; ++i) if (!active[i]) old_x[i] = old_x[i] + min_xi * (x[i] - old_x[i]);
            active[min_i] = 1;
            x[min_i] = 0.0;
        }
        Ab(n, x, y.data(), wk);
        Atx(n, y.data(), r.data(), wk);
        int64_t min_i = -1; double min_grad = 1.0;
        for (int64_t i = 0; i < np; ++i) {
            double v = r[i] - AtWd[i];
            r[i] = v * 2.0;
            if (active[i]) { if (min_i == -1 || r[i] < min_grad) { min_i = i; min_grad = r[i]; } }
        }
        if (min_i == -1 || min_grad > -0.0000001) return;
        active[min_i] = 0;
    }
}
}  // namespace

extern "C" {
void oracle_l1_ab(int64_t n, const double* b, double* d) {
    const int64_t np = n * (n - 1) / 2;
    Work w{std::vector<double>(np), std::vector<double>(np), std::vector<double>(n), std::vector<double>(n), std::vector<double>(n)};
    Ab(n, b, d, w);
}
void oracle_l1_atx(int64_t n, const double* d, double* p) {
    const int64_t np = n * (n - 1) / 2;
    Work w{std::vector<double>(np), std::vector<double>(np), std::vector<double>(n), std::vector<double>(n), std::vector<double>(n)};
    Atx(n, d, p, w);
}
double oracle_l1_tree_sum(const double* v, int64_t len) { return tree_sum(std::vector<double>(v, v + len)); }

// max_cg_iters / max_cg_calls: the budget of fnn_split_weights_budget (include/fastnn.h), 0 = none.  active_out (optional,
// npairs bytes): 1 = split held at zero by the active set when the solver returned.
int oracle_l1_split_weights(int64_t n, const double* d, double* x, int64_t* stats, int64_t max_cg_iters, int64_t max_cg_calls,
                            uint8_t* active_out) {
    const int64_t np = n * (n - 1) / 2;
    Stats st;
    std::vector<uint8_t> active(np, 0);
    unconstrainedLS(n, d, x);
    bool any_neg = false;
    for (int64_t k = 0; k < np; ++k) if (x[k] < 0.0) { any_neg = true; break; }
    if (any_neg) {
        Work wk{std::vector<double>(np), std::vector<double>(np), std::vector<double>(n), std::vector<double>(n), std::vector<double>(n)};
        activeConjugate(n, np, d, x, active, max_cg_iters > 0 ? std::min(np, max_cg_iters) : np, max_cg_calls, wk, st);
    }
    if (active_out) std::copy(active.begin(), active.end(), active_out);
    if (stats) { stats[0] = st.cg_iters; stats[1] = st.cg_calls; stats[2] = st.outer; stats[3] = st.inner; }
    return 0;
}
}
