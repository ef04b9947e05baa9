// fnn_nexus.cpp — streaming Nexus emission of the kept splits (SURVEY §8f N2).  Host only, no device calls.
//
// Produces the byte stream of OutputPrinter.NexusWithSplitsAndDistances (OutputPrinter.java:8-19: Taxa :21-32,
// Distances :34-47, Splits :49-85, st_Assumptions :87-96) from the compact result of fnn_weighted_splits / fnn_network:
// the (i, j, weight) triples of the kept splits in the live indexing of FastNN.java:409-418, split (i, j) =
// {ordering[i+1..j]}.  The reference first materialises all n(n-1)/2 BitSets (FastNN.java:405-419) and keeps the
// survivors; here a split's member list is produced only while its line is being written.
//
// Numbers are printed the way Double.toString prints them: the shortest decimal that round-trips (what JDK >= 19
// emits; older JDKs occasionally print one digit more), plain notation for 1e-3 <= |v| < 1e7, otherwise d.dddE[-]x,
// always at least one fraction digit.
#include <algorithm>
#include <atomic>
#include <charconv>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include <vector>
#include "fastnn.h"
#include "fnn_common.h"

namespace {

// Double.toString(v) into out (>= 32 bytes); returns the length (no terminator written beyond out[len] = 0).
int java_double(double v, char* out) {
    if (std::isnan(v)) { memcpy(out, "NaN", 4); return 3; }
    char* o = out;
    if (std::signbit(v)) { *o++ = '-'; v = -v; }
    if (std::isinf(v)) { memcpy(o, "Infinity", 9); return (int)(o - out) + 8; }
    if (v == 0.0) { memcpy(o, "0.0", 4); return (int)(o - out) + 3; }
    char sci[40];
    auto r = std::to_chars(sci, sci + sizeof(sci), v, std::chars_format::scientific);   // d[.ddd]e[+-]xx, shortest
    // a one-digit shortest form is widened to the two-digit decimal closest to v (the rounding interval is convex, so
    // that decimal still reads back as v): Double.MIN_VALUE prints as 4.9E-324, not 5.0E-324
    if (r.ptr > sci + 1 && sci[1] == 'e') r = std::to_chars(sci, sci + sizeof(sci), v, std::chars_format::scientific, 1);
    const char* epos = (const char*)memchr(sci, 'e', (size_t)(r.ptr - sci));
    char digits[24];
    int nd = 0;
    for (const char* p = sci; p < epos; ++p)
        if (*p != '.') digits[nd++] = *p;
    while (nd > 1 && digits[nd - 1] == '0') --nd;   // the layout below re-adds the single ".0" where it is needed
    int e10 = 0;
    {
        const char* p = epos + 1;
        const bool eneg = (*p == '-');
        if (*p == '-' || *p == '+') ++p;
        for (; p < r.ptr; ++p) e10 = e10 * 10 + (*p - '0');
        if (eneg) e10 = -e10;
    }
    if (e10 >= -3 && e10 < 7) {
        if (e10 >= 0) {
            for (int k = 0; k <= e10; ++k) *o++ = (k < nd) ? digits[k] : '0';
            *o++ = '.';
            if (nd > e10 + 1) for (int k = e10 + 1; k < nd; ++k) *o++ = digits[k];
            else *o++ = '0';
        } else {
            *o++ = '0';
            *o++ = '.';
            for (int k = 1; k < -e10; ++k) *o++ = '0';
            for (int k = 0; k < nd; ++k) *o++ = digits[k];
        }
    } else {
        *o++ = digits[0];
        *o++ = '.';
        if (nd > 1) for (int k = 1; k < nd; ++k) *o++ = digits[k];
        else *o++ = '0';
        *o++ = 'E';
        o = std::to_chars(o, o + 8, e10).ptr;
    }
    *o = 0;
    return (int)(o - out);
}

inline void put_int(std::string& s, long long v) {
    char b[24];
    s.append(b, (size_t)(std::to_chars(b, b + sizeof(b), v).ptr - b));
}

struct Sink {
    FILE* f = nullptr;
    bool own = false;
    bool failed = false;
    ~Sink() { if (f && own) fclose(f); else if (f) fflush(f); }
    void write(const std::string& s) { if (!s.empty() && fwrite(s.data(), 1, s.size(), f) != s.size()) failed = true; }
};

}  // namespace

extern "C" int fnn_java_double_to_string(double v, char* out, int64_t out_len) {
    char b[40];
    const int len = java_double(v, b);
    if (!out || out_len <= len) { fnn::set_error("fnn_java_double_to_string: need %d bytes", len + 1); return FNN_E_ARG; }
    memcpy(out, b, (size_t)len + 1);
    return FNN_OK;
}

extern "C" int fnn_write_nexus(const char* path, int64_t n, const char* names, int64_t name_stride, const double* D,
                               const int32_t* ordering, const int32_t* split_i, const int32_t* split_j, const double* weight,
                               int64_t n_splits, int threads) {
    return fnn_write_nexus_support(path, n, names, name_stride, D, ordering, split_i, split_j, weight, nullptr, 0, n_splits, threads);
}

extern "C" int fnn_write_nexus_support(const char* path, int64_t n, const char* names, int64_t name_stride, const double* D,
                                       const int32_t* ordering, const int32_t* split_i, const int32_t* split_j, const double* weight,
                                       const int32_t* support, int32_t replicates, int64_t n_splits, int threads) {
    if (n < 1 || !ordering || n_splits < 0 || (n_splits > 0 && (!split_i || !split_j || !weight)) || (names && name_stride < 1)) {
        fnn::set_error("fnn_write_nexus: bad arguments");
        return FNN_E_ARG;
    }
    if (support) {
        if (replicates < 1) { fnn::set_error("fnn_write_nexus_support: replicates %d, need >= 1", replicates); return FNN_E_ARG; }
        for (int64_t k = 0; k < n_splits; ++k)
            if (support[k] < 0 || support[k] > replicates) {
                fnn::set_error("fnn_write_nexus_support: support[%lld] = %d is outside 0..%d", (long long)k, support[k], replicates);
                return FNN_E_ARG;
            }
    }
    for (int64_t k = 0; k < n_splits; ++k)
        if (split_i[k] < 0 || split_j[k] <= split_i[k] || split_j[k] >= n) {
            fnn::set_error("fnn_write_nexus: split %lld = (%d, %d) is outside 0 <= i < j < n", (long long)k, split_i[k], split_j[k]);
            return FNN_E_ARG;
        }
    for (int64_t k = 1; k <= n; ++k)
        if (ordering[k] < 1 || ordering[k] > n) { fnn::set_error("fnn_write_nexus: ordering[%lld] = %d is not a taxon id", (long long)k, ordering[k]); return FNN_E_ARG; }
    Sink out;
    if (!path || !strcmp(path, "-")) out.f = stdout;
    else {
        out.f = fopen(path, "wb");
        out.own = true;
        if (!out.f) { fnn::set_error("cannot create %s", path); return FNN_E_IO; }
        setvbuf(out.f, nullptr, _IOFBF, 1 << 22);
    }
    int T = threads > 0 ? std::min(threads, 256) : (int)std::min<unsigned>(std::max(1u, std::thread::hardware_concurrency()), 32);

    std::string s;
    s.reserve(1 << 16);
    // ---- header + Taxa (OutputPrinter.java:9-11, :21-32)
    s += "#nexus\n\nBEGIN Taxa;\nDIMENSIONS ntax=";
    put_int(s, n);
    s += ";\nTAXLABELS\n";
    for (int64_t i = 0; i < n; ++i) {
        s += '[';
        put_int(s, i + 1);
        s += "] '";
        if (names) s.append(names + i * name_stride, strnlen(names + i * name_stride, (size_t)name_stride));
        else { s += 't'; put_int(s, i + 1); }
        s += "'\n";
        if (s.size() > (1 << 20)) { out.write(s); s.clear(); }
    }
    s += ";\nEND; [Taxa]\n\n";
    out.write(s);
    s.clear();

    // ---- Distances (:34-47): n x n values, rows formatted by the pool in batches, written in order
    if (D) {
        s += "BEGIN Distances;\nDIMENSIONS ntax=";
        put_int(s, n);
        s += ";\nFORMAT labels=no diagonal triangle=both;\nMATRIX\n";
        out.write(s);
        s.clear();
        // two row buffers: the pool formats batch b+1 while this thread writes batch b
        const int64_t batch = (int64_t)T * 8;
        std::vector<std::string> buf[2] = {std::vector<std::string>((size_t)batch), std::vector<std::string>((size_t)batch)};
        auto format_batch = [&](int64_t r0, std::vector<std::string>& rows) {
            const int64_t cnt = std::min(batch, n - r0);
            std::atomic<int64_t> next{0};
            auto body = [&]() {
                char b[40];
                for (;;) {
                    const int64_t k = next.fetch_add(1);
                    if (k >= cnt) return;
                    std::string& line = rows[(size_t)k];
                    line.clear();
                    const double* row = D + (size_t)(r0 + k) * n;
                    for (int64_t j = 0; j < n; ++j) {
                        line += ' ';
                        line.append(b, (size_t)java_double(row[j], b));
                    }
                    line += '\n';
                }
            };
            if (T <= 1 || cnt == 1) { body(); return; }
            std::vector<std::thread> pool;
            for (int t = 0; t < std::min<int64_t>(T, cnt); ++t) pool.emplace_back(body);
            for (auto& th : pool) th.join();
        };
        format_batch(0, buf[0]);
        int cur = 0;
        for (int64_t r0 = 0; r0 < n; r0 += batch, cur ^= 1) {
            const int64_t cnt = std::min(batch, n - r0);
            std::thread ahead;
            if (r0 + batch < n) ahead = std::thread(format_batch, r0 + batch, std::ref(buf[cur ^ 1]));
            for (int64_t k = 0; k < cnt && !out.failed; ++k) out.write(buf[cur][(size_t)k]);
            if (ahead.joinable()) ahead.join();
        }
        s += ";\nEND; [Distances]\n\n";
    }

    // ---- Splits (:49-85)
    s += "BEGIN Splits;\nDIMENSIONS ntax=";
    put_int(s, n);
    s += " nsplits=";
    put_int(s, n_splits);
    s += support ? ";\nFORMAT labels=no weights=yes confidences=yes intervals=no;\nPROPERTIES fit=-1.0 cyclic;\nCYCLE"
                 : ";\nFORMAT labels=no weights=yes confidences=no intervals=no;\nPROPERTIES fit=-1.0 cyclic;\nCYCLE";
    for (int64_t i = 1; i <= n; ++i) { s += ' '; put_int(s, ordering[i]); }
    s += ";\nMATRIX\n";
    std::vector<uint64_t> bits((size_t)(n + 64) / 64 + 1);
    char b[40];
    for (int64_t k = 0; k < n_splits && !out.failed; ++k) {
        const int64_t i = split_i[k], j = split_j[k];
        const int64_t card = j - i;                       // {ordering[i+1..j]}
        const int64_t size = (n - card < card) ? n - card : card;
        s += '[';
        put_int(s, k + 1);
        s += ", size=";
        put_int(s, size);
        s += "] \t ";
        s.append(b, (size_t)java_double(weight[k], b));
        s += " \t ";
        if (support) {   // the confidence column: percent of the replicates that contain the split
            s.append(b, (size_t)java_double((100.0 * (double)support[k]) / (double)replicates, b));
            s += " \t ";
        }
        // members in increasing taxon id (BitSet.nextSetBit order, :76-80)
        int lo = INT32_MAX, hi = 0;
        for (int64_t q = i + 1; q <= j; ++q) {
            const int t = ordering[q];
            bits[(size_t)t >> 6] |= 1ull << (t & 63);
            lo = std::min(lo, t);
            hi = std::max(hi, t);
        }
        for (size_t wd = (size_t)lo >> 6; wd <= ((size_t)hi >> 6); ++wd) {
            uint64_t m = bits[wd];
            bits[wd] = 0;
            while (m) {
                const int t = (int)(wd * 64) + __builtin_ctzll(m);
                m &= m - 1;
                s += ' ';
                put_int(s, t);
            }
        }
        s += ",\n";
        if (s.size() > (1 << 20)) { out.write(s); s.clear(); }
    }
    s += ";\nEND; [Splits]\n\n";
    // ---- st_Assumptions (:87-96)
    s += "BEGIN st_Assumptions;\nuptodate;\ndisttransform=NeighborNet;\nsplitstransform=EqualAngle;\nSplitsPostProcess filter=dimension value=";
    put_int(s, n);
    s += ";\n exclude  no missing;\nautolayoutnodelabels;\nEND; [st_Assumptions]\n\n";
    out.write(s);
    if (out.failed) { fnn::set_error("write to %s failed", path ? path : "stdout"); return FNN_E_IO; }
    return FNN_OK;
}
