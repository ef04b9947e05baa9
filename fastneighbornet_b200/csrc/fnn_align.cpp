// fnn_align.cpp — native nucleotide alignment loader (FASTA or sequential relaxed PHYLIP).  Host only, no device calls.
//
// The format is chosen by the first non-blank byte: '>' or ';' is FASTA, a digit is the PHYLIP header `n L`.  Codes:
// A=0 C=1 G=2 T=3 (U read as T), the IUPAC ambiguity letters R Y S W K M B D H V N and X - ? are missing data (4); case is
// ignored, whitespace inside sequence lines is skipped, and any other byte is an error naming its line and column.
//
// Layout of the work, as in fnn_phylip.cpp: the file is mmap'ed, the record starts are found in one pass (FASTA: every
// '>' at the start of a line; PHYLIP: the non-blank lines after the header), and the records are parsed by a pool of
// threads straight into the n x L code matrix.  Errors are reported for the lowest record that has one, so the message
// does not depend on the thread count.
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include "fastnn.h"
#include "fnn_common.h"
#include "fnn_hostio.h"

namespace {

constexpr uint8_t kSkip = 254, kBad = 255;

struct CodeTable {
    uint8_t t[256];
    CodeTable() {
        memset(t, kBad, sizeof(t));
        const char* states = "ACGT";
        for (int i = 0; i < 4; ++i) { t[(unsigned char)states[i]] = (uint8_t)i; t[(unsigned char)states[i] + 32] = (uint8_t)i; }
        t['U'] = t['u'] = 3;
        for (const char* p = "RYSWKMBDHVNX"; *p; ++p) { t[(unsigned char)*p] = 4; t[(unsigned char)*p + 32] = 4; }
        t['-'] = t['?'] = 4;
        t[' '] = kSkip;
        for (int c = 9; c <= 13; ++c) t[c] = kSkip;
    }
};
const CodeTable kCode;

inline bool is_ws(unsigned char c) { return c == ' ' || (c >= 9 && c <= 13); }

// 1-based line and column of p (error path only)
void locate(const char* base, const char* p, long long* line, long long* col) {
    long long ln = 1;
    const char* ls = base;
    for (const char* q = base; q < p;) {
        const char* nl = (const char*)memchr(q, '\n', (size_t)(p - q));
        if (!nl) break;
        ++ln;
        ls = q = nl + 1;
    }
    *line = ln;
    *col = (long long)(p - ls) + 1;
}

std::string show_byte(unsigned char c) {
    char b[16];
    if (c >= 33 && c < 127) snprintf(b, sizeof(b), "'%c'", c);
    else snprintf(b, sizeof(b), "byte 0x%02x", c);
    return b;
}

// Codes of the sequence characters in [s, e): stores the first `cap` of them to out (if non-null) and returns how many there
// are, or -1 with *bad at the first byte that is neither a code nor whitespace.  fasta: lines starting with ';' are skipped.
int64_t scan_seq(const char* s, const char* e, bool fasta, uint8_t* out, int64_t cap, const char** bad) {
    int64_t count = 0;
    while (s < e) {
        const char* le = fasta ? fnn::line_end(s, e) : e;
        if (!(fasta && *s == ';')) {
            for (const char* p = s; p < le; ++p) {
                const uint8_t c = kCode.t[(unsigned char)*p];
                if (c == kSkip) continue;
                if (c == kBad) { *bad = p; return -1; }
                if (out && count < cap) out[count] = c;
                ++count;
            }
        }
        s = le < e ? le + 1 : e;
    }
    return count;
}

struct Record {
    const char* name;      // name text [name, name_end)
    const char* name_end;
    const char* seq;       // sequence text [seq, end)
    const char* end;
};

void copy_name(const Record& r, char* dst, int64_t stride) {
    const size_t k = std::min<size_t>((size_t)(r.name_end - r.name), (size_t)stride - 1);
    memcpy(dst, r.name, k);
    dst[k] = 0;
}

std::string name_of(const Record& r) { return std::string(r.name, std::min<size_t>((size_t)(r.name_end - r.name), 64)); }

struct Parsed {
    bool fasta = false;
    long long n_header = 0, sites_header = 0;   // PHYLIP header
    std::vector<Record> recs;
};

// PHYLIP header `n L` -> 0, or FNN_E_IO
int parse_phylip_header(const char* s, const char* e, long long* n, long long* sites) {
    long long v[2] = {0, 0};
    int got = 0;
    const char* p = s;
    while (got < 2) {
        while (p < e && is_ws((unsigned char)*p)) ++p;
        int digits = 0;
        while (p < e && *p >= '0' && *p <= '9' && digits <= 12) { v[got] = v[got] * 10 + (*p - '0'); ++p; ++digits; }
        if (!digits || (p < e && !is_ws((unsigned char)*p))) return FNN_E_IO;
        ++got;
    }
    while (p < e && is_ws((unsigned char)*p)) ++p;
    if (p != e) return FNN_E_IO;
    *n = v[0];
    *sites = v[1];
    return FNN_OK;
}

void record_error(const char* path, const char* base, const Parsed& P, int64_t r, int64_t count, const char* bad, int64_t sites);

// Format detection and the record starts (one pass over the file).
int find_records(const char* path, const char* base, const char* end, Parsed* out) {
    const char* p = base;
    while (p < end && is_ws((unsigned char)*p)) ++p;
    if (p == end) { fnn::set_error("%s: no sequences", path); return FNN_E_IO; }
    if (*p == '>' || *p == ';') {
        out->fasta = true;
        for (const char* q = p; q < end;) {
            const char* g = (const char*)memchr(q, '>', (size_t)(end - q));
            if (!g) break;
            if (g == base || g[-1] == '\n') {
                const char* he = fnn::line_end(g, end);
                const char* ne = g + 1;
                while (ne < he && !is_ws((unsigned char)*ne)) ++ne;
                if (!out->recs.empty()) out->recs.back().end = g;
                out->recs.push_back({g + 1, ne, he < end ? he + 1 : end, end});
            }
            q = g + 1;
        }
        if (out->recs.empty()) { fnn::set_error("%s: no sequences", path); return FNN_E_IO; }
        return FNN_OK;
    }
    if (*p < '0' || *p > '9') {
        long long line, col;
        locate(base, p, &line, &col);
        fnn::set_error("%s: line %lld starts with %s; expected '>' (FASTA) or a PHYLIP header `n L`", path, line,
                       show_byte((unsigned char)*p).c_str());
        return FNN_E_IO;
    }
    const char* he = fnn::line_end(p, end);
    if (parse_phylip_header(p, he, &out->n_header, &out->sites_header)) {
        long long line, col;
        locate(base, p, &line, &col);
        fnn::set_error("%s: line %lld is not a PHYLIP header `n L`", path, line);
        return FNN_E_IO;
    }
    if (out->n_header < 1) { fnn::set_error("%s: no sequences (header says %lld taxa)", path, out->n_header); return FNN_E_IO; }
    if (out->sites_header < 1 || out->sites_header > INT32_MAX) {
        fnn::set_error("%s: header says %lld sites; an alignment has 1 .. 2^31-1 sites", path, out->sites_header);
        return FNN_E_IO;
    }
    long long extra_line = 0;
    for (const char* s = he < end ? he + 1 : end; s < end;) {
        const char* e = fnn::line_end(s, end);
        const char* t = s;
        while (t < e && is_ws((unsigned char)*t)) ++t;
        if (t < e) {   // not blank
            if ((long long)out->recs.size() == out->n_header) { extra_line = 1; out->recs.push_back({t, t, t, e}); break; }
            const char* ne = t;
            while (ne < e && !is_ws((unsigned char)*ne)) ++ne;
            out->recs.push_back({t, ne, ne, e});
        }
        s = e < end ? e + 1 : end;
    }
    if (extra_line) {
        // interleaved PHYLIP: its first block is shorter than L, so name that; otherwise the file simply has too many lines
        const char* bad = nullptr;
        const int64_t first = scan_seq(out->recs[0].seq, out->recs[0].end, false, nullptr, 0, &bad);
        if (first != out->sites_header) { record_error(path, base, *out, 0, first, bad, out->sites_header); return FNN_E_IO; }
        long long line, col;
        locate(base, out->recs.back().name, &line, &col);
        fnn::set_error("%s: header says %lld taxa, but line %lld holds a further sequence (interleaved PHYLIP is not read)", path,
                       out->n_header, line);
        return FNN_E_IO;
    }
    if ((long long)out->recs.size() != out->n_header) {
        fnn::set_error("%s: header says %lld taxa, the file has %lld sequence lines", path, out->n_header, (long long)out->recs.size());
        return FNN_E_IO;
    }
    return FNN_OK;
}

// the error of record r, whose scan returned `count` (or -1 with `bad`) against the expected `sites`
void record_error(const char* path, const char* base, const Parsed& P, int64_t r, int64_t count, const char* bad, int64_t sites) {
    const Record& rec = P.recs[(size_t)r];
    long long line, col;
    if (count < 0) {
        locate(base, bad, &line, &col);
        fnn::set_error("%s: line %lld, column %lld: %s is not a nucleotide or missing-data code (taxon %lld '%s')", path, line, col,
                       show_byte((unsigned char)*bad).c_str(), (long long)r + 1, name_of(rec).c_str());
        return;
    }
    locate(base, rec.name, &line, &col);
    if (count == 0) {
        fnn::set_error("%s: taxon %lld '%s' (line %lld) has an empty sequence", path, (long long)r + 1, name_of(rec).c_str(), line);
        return;
    }
    fnn::set_error("%s: taxon %lld '%s' (line %lld) has %lld sites, expected %lld%s", path, (long long)r + 1, name_of(rec).c_str(), line,
                   (long long)count, (long long)sites, P.fasta ? "" : " (interleaved PHYLIP is not read)");
}

}  // namespace

extern "C" int fnn_alignment_size(const char* path, int64_t* n_out, int64_t* sites_out) {
    if (!path || !n_out || !sites_out) { fnn::set_error("fnn_alignment_size: null argument"); return FNN_E_ARG; }
    fnn::Mapped f;
    int rc = f.open_(path);
    if (rc) return rc;
    Parsed P;
    rc = find_records(path, f.p, f.p + f.len, &P);
    if (rc) return rc;
    int64_t sites = P.sites_header;
    if (P.fasta) {   // the first record's length; fnn_read_alignment holds every other record to it
        const char* bad = nullptr;
        sites = scan_seq(P.recs[0].seq, P.recs[0].end, true, nullptr, 0, &bad);
        if (sites <= 0) { record_error(path, f.p, P, 0, sites, bad, 0); return FNN_E_IO; }
        if (sites > INT32_MAX) { fnn::set_error("%s: %lld sites; an alignment has at most 2^31-1", path, (long long)sites); return FNN_E_IO; }
    }
    *n_out = (int64_t)P.recs.size();
    *sites_out = sites;
    return FNN_OK;
}

extern "C" int fnn_read_alignment(const char* path, int64_t n, int64_t sites, uint8_t* codes, char* names, int64_t name_stride,
                                  int threads) {
    if (!path || !codes || n < 1 || sites < 1 || (names && name_stride < 1)) {
        fnn::set_error("fnn_read_alignment: need path, n >= 1, sites >= 1, an n*sites code array and name_stride >= 1 with names");
        return FNN_E_ARG;
    }
    fnn::Mapped f;
    int rc = f.open_(path);
    if (rc) return rc;
    Parsed P;
    rc = find_records(path, f.p, f.p + f.len, &P);
    if (rc) return rc;
    const int64_t nf = (int64_t)P.recs.size();
    if (nf != n || (!P.fasta && P.sites_header != sites)) {
        fnn::set_error("%s: %lld taxa%s, caller says %lld taxa x %lld sites", path, (long long)nf,
                       P.fasta ? "" : (" x " + std::to_string(P.sites_header) + " sites").c_str(), (long long)n, (long long)sites);
        return FNN_E_ARG;
    }
    std::vector<int64_t> counts((size_t)n);
    std::vector<const char*> bads((size_t)n, nullptr);
    constexpr int64_t RB = 16;
    std::atomic<int64_t> next{0};
    fnn::run_pool(fnn::pick_threads(threads), [&](int) {
        for (;;) {
            const int64_t b = next.fetch_add(1);
            if (b * RB >= n) return;
            for (int64_t r = b * RB; r < std::min(n, (b + 1) * RB); ++r) {
                const Record& rec = P.recs[(size_t)r];
                counts[(size_t)r] = scan_seq(rec.seq, rec.end, P.fasta, codes + (size_t)r * (size_t)sites, sites, &bads[(size_t)r]);
                if (names) copy_name(rec, names + (size_t)r * (size_t)name_stride, name_stride);
            }
        }
    });
    for (int64_t r = 0; r < n; ++r) {
        if (counts[(size_t)r] != sites) {
            record_error(path, f.p, P, r, counts[(size_t)r], bads[(size_t)r], sites);
            return FNN_E_IO;
        }
    }
    return FNN_OK;
}
