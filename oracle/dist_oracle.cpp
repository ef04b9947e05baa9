// dist_oracle.cpp — CPU restatement of the alignment distances of fnn_distances / fnn_ctx_load_alignment (include/fastnn.h,
// DESIGN.md §4.4).  TEST INFRASTRUCTURE ONLY.
//
// It counts v, m and s with a plain per-pair, per-site loop over the code bytes and shares none of the device's bit-plane
// packing or popcount logic; only the logarithm (csrc/fnn_log.h) is the same code on both sides.  It computes the listed
// rows only, so a production size can be held to it on a sample of rows.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <thread>
#include <vector>
#include "../fastneighbornet_b200/csrc/fnn_log.h"

namespace {

// d of the model, or NaN and *undef when v = 0 or an argument of a log is <= 0
double model_distance(int model, int64_t v, int64_t m, int64_t s, bool* undef) {
    *undef = false;
    if (v == 0) { *undef = true; return NAN; }
    const double dv = (double)v;
    double d;
    if (model == 0) {
        d = (double)m / dv;
    } else if (model == 1) {
        const double p = (double)m / dv;
        const double arg = 1.0 - p / 0.75;
        if (arg <= 0.0) { *undef = true; return NAN; }
        d = -0.75 * fnn_log(arg);
    } else {
        const double P = (double)s / dv, Q = (double)(m - s) / dv;
        const double a1 = (1.0 - 2.0 * P) - Q, a2 = 1.0 - 2.0 * Q;
        if (a1 <= 0.0 || a2 <= 0.0) { *undef = true; return NAN; }
        d = (-0.5 * fnn_log(a1)) - (0.25 * fnn_log(a2));
    }
    if (d == 0.0) d = 0.0;
    return d;
}

}  // namespace

extern "C" void oracle_fnn_log(const double* x, int64_t count, double* out) {
    for (int64_t k = 0; k < count; ++k) out[k] = fnn_log(x[k]);
}

// codes: n x L row-major (0..4).  rows[nrows]: the rows to compute, D_rows_out[nrows * n].  undefined_value NaN leaves NaN in
// undefined entries, anything else is stored there.  first_undefined_out[5] = {i, j, v, m, s} of the undefined pair i < j with
// the lowest (i, j) among the computed rows, i = -1 if there is none.  Returns 0, or -1 for a bad argument (a code > 4).
extern "C" int oracle_distances(const uint8_t* codes, int64_t n, int64_t L, int model, double undefined_value, const int64_t* rows,
                                int64_t nrows, double* D_rows_out, int64_t* first_undefined_out) {
    if (!codes || n < 1 || L < 1 || model < 0 || model > 2 || !rows || nrows < 0 || !D_rows_out) return -1;
    for (int64_t k = 0; k < n * L; ++k)
        if (codes[k] > 4) return -1;
    for (int64_t r = 0; r < nrows; ++r)
        if (rows[r] < 0 || rows[r] >= n) return -1;
    const unsigned hc = std::thread::hardware_concurrency();
    const int T = (int)std::max<unsigned>(1, std::min<unsigned>(hc ? hc : 1, 64));
    std::vector<int64_t> first((size_t)T * 5, -1);
    std::atomic<int64_t> next{0};
    auto body = [&](int t) {
        int64_t* f = &first[(size_t)t * 5];
        for (;;) {
            const int64_t r = next.fetch_add(1);
            if (r >= nrows) return;
            const int64_t i = rows[r];
            const uint8_t* x = codes + i * L;
            double* out = D_rows_out + r * n;
            for (int64_t j = 0; j < n; ++j) {
                if (j == i) { out[j] = 0.0; continue; }
                const uint8_t* y = codes + j * L;
                int32_t v = 0, m = 0, s = 0;   // L <= 2^31-1
                for (int64_t k = 0; k < L; ++k) {
                    const unsigned a = x[k], b = y[k];
                    const int32_t both = (a < 4) & (b < 4);
                    v += both;
                    m += both & (a != b);
                    s += both & ((a ^ b) == 2);   // A<->G (0,2) and C<->T (1,3)
                }
                bool undef;
                const double d = model_distance(model, v, m, s, &undef);
                if (!undef) { out[j] = d; continue; }
                out[j] = std::isnan(undefined_value) ? d : undefined_value;
                const int64_t lo = std::min(i, j), hi = std::max(i, j);
                if (f[0] < 0 || lo < f[0] || (lo == f[0] && hi < f[1])) { f[0] = lo; f[1] = hi; f[2] = v; f[3] = m; f[4] = s; }
            }
        }
    };
    std::vector<std::thread> pool;
    for (int t = 0; t < T; ++t) pool.emplace_back(body, t);
    for (auto& th : pool) th.join();
    int64_t* best = first_undefined_out;
    if (best) {
        for (int k = 0; k < 5; ++k) best[k] = -1;
        for (int t = 0; t < T; ++t) {
            const int64_t* f = &first[(size_t)t * 5];
            if (f[0] >= 0 && (best[0] < 0 || f[0] < best[0] || (f[0] == best[0] && f[1] < best[1])))
                for (int k = 0; k < 5; ++k) best[k] = f[k];
        }
    }
    return 0;
}
