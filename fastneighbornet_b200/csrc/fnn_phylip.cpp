// fnn_phylip.cpp — native Phylip distance-matrix loader (SURVEY §8f N1).  Host only, no device calls.
//
// Replaces the reference's two passes over the file (FastNN.java:270-276 for the header, DistancesAndNames.java:43-132
// for the rows) and its packed-triangle -> double[n][n] copy (FastNN.java:297-312).  Conventions kept from the Java:
//   * line 1: the taxon count after stripping ALL whitespace (FastNN.java:272-274);
//   * every further line: `name v v v ...`; the name is everything up to the first ' ' (line.split(" ")[0], :62-66), the
//     values are the non-empty pieces of the rest split on ' ' and then on '\t' (:68-76);
//   * only the first `row` values of row `row` are consumed (:78-83), so lower-triangular and square files both load;
//   * reading stops after n rows (names[row] throws at row == n, :64-67).
// Double.valueOf and strtod are both correctly rounded, so every parsed value is the same double as in the JVM.
//
// Layout of the work: the file is mmap'ed, the n row starts are found with one memchr pass, the rows are parsed by a
// pool of threads (rows handed out in blocks, row r costs r values), and the lower triangle is then mirrored into the
// upper one tile by tile so that neither pass makes strided single-element writes.
#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>
#include "fastnn.h"
#include "fnn_common.h"
#include "fnn_hostio.h"

namespace {

using fnn::Mapped;
using fnn::line_end;
using fnn::pick_threads;
using fnn::run_pool;

// header line -> taxon count (all whitespace stripped, then Integer.parseInt)
int parse_header(const char* s, const char* e, long long* n_out) {
    long long v = 0;
    int digits = 0;
    for (; s < e; ++s) {
        const unsigned char ch = (unsigned char)*s;
        if (ch == ' ' || (ch >= 9 && ch <= 13)) continue;
        if (ch < '0' || ch > '9' || digits > 12) return FNN_E_IO;
        v = v * 10 + (ch - '0');
        ++digits;
    }
    if (!digits) return FNN_E_IO;
    *n_out = v;
    return FNN_OK;
}

const double kPow10[23] = {1e0,  1e1,  1e2,  1e3,  1e4,  1e5,  1e6,  1e7,  1e8,  1e9,  1e10, 1e11,
                           1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};

#if defined(__x86_64__) && defined(__LDBL_MANT_DIG__) && __LDBL_MANT_DIG__ == 64
#define FNN_HAVE_X87 1
// 10^0 .. 10^27 are exact in the x87 format (5^27 < 2^64)
struct Pow10L {
    long double v[28];
    Pow10L() { v[0] = 1.0L; for (int i = 1; i < 28; ++i) v[i] = v[i - 1] * 10.0L; }
};
const Pow10L kPow10L;
#endif

// One value token [s, e).  Path 1 (Clinger): at most 15 significant digits and |decimal exponent| <= 22 -> the integer
// mantissa and the power of ten are both exact doubles, so one multiply or divide rounds correctly.  Path 2 (up to 19
// digits, |exponent| <= 27, the 17-digit round-trip output of most writers): mantissa and power are exact in the 64-bit
// x87 format, the quotient/product is within half a unit of its 64th bit, so rounding it to 53 bits is the correct
// rounding of the decimal unless it sits within one such unit of a double midpoint (low 11 bits 0x3FF..0x401) - those
// rare tokens, and everything else (huge exponents, inf/nan, hex), go to strtod, which is correctly rounded too.
double parse_value(const char* s, const char* e) {
    const char* p = s;
    bool neg = false;
    if (p < e && (*p == '-' || *p == '+')) { neg = (*p == '-'); ++p; }
    uint64_t w = 0;
    int sig = 0, exp10 = 0;
    bool any = false, ok = true;
    for (; p < e && *p >= '0' && *p <= '9'; ++p) {
        any = true;
        if (sig > 0 || *p != '0') { if (sig < 19) { w = w * 10 + (uint64_t)(*p - '0'); ++sig; } else { ok = false; } }
    }
    if (p < e && *p == '.') {
        ++p;
        for (; p < e && *p >= '0' && *p <= '9'; ++p) {
            any = true;
            if (sig > 0 || *p != '0') { if (sig < 19) { w = w * 10 + (uint64_t)(*p - '0'); ++sig; } else { ok = false; } }
            --exp10;
        }
    }
    if (any && p < e && (*p == 'e' || *p == 'E')) {
        const char* q = p + 1;
        bool eneg = false;
        if (q < e && (*q == '-' || *q == '+')) { eneg = (*q == '-'); ++q; }
        int ev = 0, ed = 0;
        for (; q < e && *q >= '0' && *q <= '9'; ++q) { if (ev < 100000) ev = ev * 10 + (*q - '0'); ++ed; }
        if (ed) { exp10 += eneg ? -ev : ev; p = q; }
    }
    if (any && ok && p == e && sig <= 15 && exp10 >= -22 && exp10 <= 22) {
        double v = (double)w;
        v = (exp10 < 0) ? v / kPow10[-exp10] : v * kPow10[exp10];
        return neg ? -v : v;
    }
#ifdef FNN_HAVE_X87
    if (any && ok && p == e && sig <= 19 && w != 0 && exp10 >= -27 && exp10 <= 27) {
        const long double q = (exp10 < 0) ? (long double)w / kPow10L.v[-exp10] : (long double)w * kPow10L.v[exp10];
        uint64_t mant;
        memcpy(&mant, &q, sizeof(mant));
        const unsigned low = (unsigned)(mant & 0x7FF);
        if (low < 0x3FF || low > 0x401) {
            const double v = (double)q;
            return neg ? -v : v;
        }
    }
#endif
    char small[64];
    const size_t len = (size_t)(e - s);
    if (len < sizeof(small)) {
        memcpy(small, s, len);
        small[len] = 0;
        return strtod(small, nullptr);
    }
    return strtod(std::string(s, len).c_str(), nullptr);
}

// Parses row `row` from the line [s, e): writes D[row][0..row).  Returns the number of values consumed.
int64_t parse_row(const char* s, const char* e, int64_t row, double* out, char* name, int64_t name_stride) {
    if (e > s && e[-1] == '\r') --e;
    const char* sp = (const char*)memchr(s, ' ', (size_t)(e - s));
    const char* name_end = sp ? sp : e;
    if (name && name_stride > 0) {
        const size_t k = std::min<size_t>((size_t)(name_end - s), (size_t)name_stride - 1);
        memcpy(name, s, k);
        name[k] = 0;
    }
    int64_t col = 0;
    const char* p = name_end;
    while (col < row && p < e) {
        while (p < e && (*p == ' ' || *p == '\t')) ++p;
        if (p >= e) break;
        const char* t = p;
        while (p < e && *p != ' ' && *p != '\t') ++p;
        out[col++] = parse_value(t, p);
    }
    return col;
}

}  // namespace

extern "C" int fnn_phylip_taxa(const char* path, int64_t* n_out) {
    if (!path || !n_out) { fnn::set_error("fnn_phylip_taxa: null argument"); return FNN_E_ARG; }
    Mapped f;
    int rc = f.open_(path);
    if (rc) return rc;
    long long n = 0;
    if (parse_header(f.p, line_end(f.p, f.p + f.len), &n)) { fnn::set_error("%s: first line is not a taxon count", path); return FNN_E_IO; }
    *n_out = n;
    return FNN_OK;
}

extern "C" int fnn_read_phylip(const char* path, int64_t n, double* D, char* names, int64_t name_stride, int threads) {
    if (!path || !D || n < 1) { fnn::set_error("fnn_read_phylip: need path, n >= 1 and an n*n output"); return FNN_E_ARG; }
    Mapped f;
    int rc = f.open_(path);
    if (rc) return rc;
    const char* end = f.p + f.len;
    const char* he = line_end(f.p, end);
    long long n_file = 0;
    if (parse_header(f.p, he, &n_file)) { fnn::set_error("%s: first line is not a taxon count", path); return FNN_E_IO; }
    if (n_file != n) { fnn::set_error("%s: header says %lld taxa, caller says %lld", path, n_file, (long long)n); return FNN_E_ARG; }

    // row extents: one sequential memchr pass (memory speed), stops after n lines
    std::vector<const char*> row_s((size_t)n), row_e((size_t)n);
    int64_t rows = 0;
    for (const char* s = (he < end) ? he + 1 : end; rows < n && s < end;) {
        const char* e = line_end(s, end);
        if (e == s || (e == s + 1 && *s == '\r')) break;   // blank line: end of data
        row_s[(size_t)rows] = s;
        row_e[(size_t)rows] = e;
        ++rows;
        s = (e < end) ? e + 1 : end;
    }
    if (rows < n) { fnn::set_error("%s: %lld rows, expected %lld", path, (long long)rows, (long long)n); return FNN_E_IO; }

    const int T = pick_threads(threads);
    // rows are parsed from the bottom up in blocks: the long rows go first, so the tail of the schedule is cheap
    constexpr int64_t RB = 8;
    std::atomic<int64_t> next_block{0};
    std::atomic<int64_t> bad_row{INT64_MAX};
    const int64_t nblocks = (n + RB - 1) / RB;
    run_pool(T, [&](int) {
        for (;;) {
            const int64_t b = next_block.fetch_add(1);
            if (b >= nblocks) return;
            const int64_t hi = n - b * RB, lo = std::max<int64_t>(0, hi - RB);
            for (int64_t r = hi - 1; r >= lo; --r) {
                const int64_t got = parse_row(row_s[(size_t)r], row_e[(size_t)r], r, D + (size_t)r * n, names ? names + (size_t)r * name_stride : nullptr, name_stride);
                D[(size_t)r * n + r] = 0.0;
                if (got < r) {
                    int64_t cur = bad_row.load();
                    while (r < cur && !bad_row.compare_exchange_weak(cur, r)) {}
                }
            }
        }
    });
    if (bad_row.load() != INT64_MAX) {
        fnn::set_error("%s: row %lld has fewer than %lld lower-triangle values", path, (long long)bad_row.load(), (long long)bad_row.load());
        return FNN_E_IO;
    }

    // mirror lower -> upper, 64 x 64 tiles (reads along rows, writes along rows of the transposed tile)
    constexpr int64_t TB = 64;
    const int64_t nt = (n + TB - 1) / TB;
    std::atomic<int64_t> next_tile{0};
    run_pool(T, [&](int) {
        for (;;) {
            const int64_t bi = next_tile.fetch_add(1);
            if (bi >= nt) return;
            const int64_t r0 = bi * TB, r1 = std::min(n, r0 + TB);
            for (int64_t bj = 0; bj <= bi; ++bj) {
                const int64_t c0 = bj * TB, c1 = std::min(n, c0 + TB);
                for (int64_t c = c0; c < c1; ++c) {
                    double* dst = D + (size_t)c * n;
                    for (int64_t r = std::max(r0, c + 1); r < r1; ++r) dst[r] = D[(size_t)r * n + c];
                }
            }
        }
    });
    return FNN_OK;
}
