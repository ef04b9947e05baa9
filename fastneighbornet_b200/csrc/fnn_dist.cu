// fnn_dist.cu — pairwise distances of a nucleotide alignment on the device (P, JC69, K2P; pairwise deletion), written
// straight into a device matrix: the context's own (fnn_ctx_load_alignment, fnn_bootstrap) or a scratch buffer copied back to
// the host (fnn_distances).  DESIGN.md §4.4.  DistJob (fnn_common.h) uploads the codes once; a bootstrap replicate then
// packs its planes through its list of drawn columns.
//
//   k_pack   codes (uint8, n x L, 0..4) -> three bit-planes per 64-site word and taxon.  With A=00 G=01 C=10 T=11 (hi, lo):
//            hi = pyrimidine, lo = G or T, ok = the site holds a state.  ok is 0 past L and for padding
//            taxa, so no count ever sees them.  Layout planes[(w * 3 + plane) * np + taxon], np = n rounded up to TM.
//   k_pairs  one CTA per lower-triangle tile (ti >= tj) of TM x TM pairs, a K-loop over the words staged through shared
//            memory with cp.async double buffering, an MT x MT register micro-tile of counters per thread:
//              v += popc(okx & oky)                      comparable sites
//              m += popc(((hx ^ hy) | (lx ^ ly)) & ok)    differences
//              q += popc((hx ^ hy) & ok)                 transversions (K2P only); s = m - q
//            then the model formula, D[i][j] directly and D[j][i] through a transposed shared-memory tile, so both stores
//            are row-contiguous.  The first undefined pair i < j is the minimum of i * n + j (64-bit atomicMin).
// Every formula is binary64 with the library's --fmad=false; fnn_log (csrc/fnn_log.h) is the logarithm the CPU oracle
// (oracle/dist_oracle.cpp) uses too, so the device and the oracle agree bit for bit.
#include <cuda_runtime.h>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>
#include "fastnn.h"
#include "fnn_common.h"
#include "fnn_log.h"

namespace {

constexpr int TM = 64;        // taxa per tile side
constexpr int BK = 8;         // 64-site words per pipeline stage
constexpr int THREADS = 256;  // 16 x 16 threads, MT x MT pairs each
constexpr int MT = 4;
constexpr int PLANES = 3;     // hi, lo, ok
static_assert(16 * MT == TM, "micro-tile layout");

const char* model_name(int32_t model) { return model == FNN_DIST_P ? "p" : (model == FNN_DIST_JC69 ? "jc69" : "k2p"); }

// one warp per (taxon, word): each lane maps two sites, three ballots give the word's planes.  sites (optional, L entries):
// site s of the packed alignment is column sites[s] of codes (a bootstrap replicate); NULL = column s.
__global__ void k_pack(const uint8_t* __restrict__ codes, int64_t n, int64_t L, int64_t W, int64_t np, const int32_t* __restrict__ sites,
                       unsigned long long* __restrict__ planes, int* __restrict__ bad) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x / 32);
    for (int64_t u = (int64_t)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32; u < n * W; u += warps) {
        const int64_t t = u / W, w = u - t * W;
        const int64_t s0 = w * 64 + lane, s1 = s0 + 32;
        const unsigned c0 = s0 < L ? codes[t * L + (sites ? sites[s0] : s0)] : 4u;
        const unsigned c1 = s1 < L ? codes[t * L + (sites ? sites[s1] : s1)] : 4u;
        if (c0 > 4u || c1 > 4u) atomicOr(bad, 1);
        const bool ok0 = c0 < 4u, ok1 = c1 < 4u;
        const unsigned hi0 = __ballot_sync(0xffffffffu, ok0 && (c0 & 1u)), hi1 = __ballot_sync(0xffffffffu, ok1 && (c1 & 1u));
        const unsigned lo0 = __ballot_sync(0xffffffffu, ok0 && c0 >= 2u), lo1 = __ballot_sync(0xffffffffu, ok1 && c1 >= 2u);
        const unsigned k0 = __ballot_sync(0xffffffffu, ok0), k1 = __ballot_sync(0xffffffffu, ok1);
        if (lane == 0) {
            planes[(w * PLANES + 0) * np + t] = (unsigned long long)hi0 | ((unsigned long long)hi1 << 32);
            planes[(w * PLANES + 1) * np + t] = (unsigned long long)lo0 | ((unsigned long long)lo1 << 32);
            planes[(w * PLANES + 2) * np + t] = (unsigned long long)k0 | ((unsigned long long)k1 << 32);
        }
    }
}

// d(v, m, q) of §1 of include/fastnn.h; *undef when v = 0 or an argument of a log is <= 0
template <int MODEL>
__device__ __forceinline__ double dist_value(int v, int m, int q, bool* undef) {
    *undef = false;
    if (v == 0) { *undef = true; return 0.0; }
    const double dv = (double)v;
    double d;
    if (MODEL == FNN_DIST_P) {
        d = (double)m / dv;
    } else if (MODEL == FNN_DIST_JC69) {
        const double p = (double)m / dv;
        const double a = 1.0 - p / 0.75;
        if (!(a > 0.0)) { *undef = true; return 0.0; }
        d = -0.75 * fnn_log(a);
    } else {
        const double P = (double)(m - q) / dv, Q = (double)q / dv;
        const double a1 = (1.0 - 2.0 * P) - Q, a2 = 1.0 - 2.0 * Q;
        if (!(a1 > 0.0) || !(a2 > 0.0)) { *undef = true; return 0.0; }
        d = (-0.5 * fnn_log(a1)) - (0.25 * fnn_log(a2));
    }
    return d == 0.0 ? 0.0 : d;   // -0.0 (m = 0 through -0.75 * log(1)) is stored as +0.0
}

struct __align__(16) Stage {
    unsigned long long w[BK][PLANES][2][TM];   // [word][plane][x/y side][taxon]
};
static_assert(2 * sizeof(Stage) >= sizeof(double) * TM * (TM + 1), "the transposed tile reuses the stages");

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}

template <int MODEL>
__global__ void __launch_bounds__(THREADS) k_pairs(const unsigned long long* __restrict__ planes, int64_t np, int64_t stages,
                                                  int n, double* __restrict__ D, int64_t ld, double undef_value, int fail,
                                                  unsigned long long* __restrict__ first_undef) {
    __shared__ Stage sm[2];
    const int64_t b = blockIdx.x;
    int64_t ti = (int64_t)((sqrt(8.0 * (double)b + 1.0) - 1.0) * 0.5);
    while (ti * (ti + 1) / 2 > b) --ti;
    while ((ti + 1) * (ti + 2) / 2 <= b) ++ti;
    const int64_t tj = b - ti * (ti + 1) / 2;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;

    auto load = [&](int64_t s, int buf) {
        // 48 rows (word, plane, side) of TM taxa = 32 chunks of 16 bytes each
        for (int idx = tid; idx < BK * PLANES * 2 * (TM / 2); idx += THREADS) {
            const int r = idx / (TM / 2), c = idx % (TM / 2);
            const int w = r / (PLANES * 2), pl = (r / 2) % PLANES, side = r & 1;
            const unsigned long long* src = planes + ((s * BK + w) * PLANES + pl) * np + (side ? tj : ti) * TM + 2 * c;
            cp_async16(&sm[buf].w[w][pl][side][2 * c], src);
        }
        asm volatile("cp.async.commit_group;\n" ::);
    };

    int v[MT][MT], m[MT][MT], q[MT][MT];
#pragma unroll
    for (int a = 0; a < MT; ++a)
#pragma unroll
        for (int c = 0; c < MT; ++c) v[a][c] = m[a][c] = q[a][c] = 0;

    load(0, 0);
    for (int64_t s = 0; s < stages; ++s) {
        const int buf = (int)(s & 1);
        if (s + 1 < stages) {
            load(s + 1, buf ^ 1);
            asm volatile("cp.async.wait_group 1;\n" ::);
        } else {
            asm volatile("cp.async.wait_group 0;\n" ::);
        }
        __syncthreads();
#pragma unroll 2
        for (int w = 0; w < BK; ++w) {
            unsigned long long xh[MT], xl[MT], xo[MT];
#pragma unroll
            for (int a = 0; a < MT; ++a) {
                xh[a] = sm[buf].w[w][0][0][ty + 16 * a];
                xl[a] = sm[buf].w[w][1][0][ty + 16 * a];
                xo[a] = sm[buf].w[w][2][0][ty + 16 * a];
            }
#pragma unroll
            for (int c = 0; c < MT; ++c) {
                const unsigned long long yh = sm[buf].w[w][0][1][tx + 16 * c];
                const unsigned long long yl = sm[buf].w[w][1][1][tx + 16 * c];
                const unsigned long long yo = sm[buf].w[w][2][1][tx + 16 * c];
#pragma unroll
                for (int a = 0; a < MT; ++a) {
                    const unsigned long long ok = xo[a] & yo, tv = xh[a] ^ yh;
                    v[a][c] += __popcll(ok);
                    m[a][c] += __popcll((tv | (xl[a] ^ yl)) & ok);
                    if (MODEL == FNN_DIST_K2P) q[a][c] += __popcll(tv & ok);
                }
            }
        }
        __syncthreads();
    }

    // epilogue: the stages are free (the last __syncthreads above), the transposed tile reuses them
    double* T = reinterpret_cast<double*>(&sm[0]);
    const bool diag = ti == tj;
#pragma unroll
    for (int a = 0; a < MT; ++a) {
#pragma unroll
        for (int c = 0; c < MT; ++c) {
            const int64_t i = ti * TM + ty + 16 * a, j = tj * TM + tx + 16 * c;
            bool undef;
            double d = dist_value<MODEL>(v[a][c], m[a][c], q[a][c], &undef);
            if (i == j) {
                d = 0.0;
            } else if (undef) {
                d = undef_value;
                if (fail && i < n && j < n)
                    atomicMin(first_undef, (unsigned long long)(i < j ? i * n + j : j * n + i));
            }
            if (i < n && j < n) D[i * ld + j] = d;
            if (!diag) T[(tx + 16 * c) * (TM + 1) + ty + 16 * a] = d;
        }
    }
    if (!diag) {
        __syncthreads();
        for (int e = tid; e < TM * TM; e += THREADS) {
            const int jj = e / TM, ii = e % TM;
            const int64_t i = ti * TM + ii, j = tj * TM + jj;
            if (i < n && j < n) D[j * ld + i] = T[jj * (TM + 1) + ii];
        }
    }
}

}  // namespace

int fnn_dist_check_args_(const char* who, const uint8_t* codes, int64_t n, int64_t sites, int32_t model, double undef) {
    if (!codes || n < 1 || n > 2000000 || sites < 1 || sites > INT32_MAX) {
        fnn::set_error("%s: need codes, 1 <= n <= 2000000 and 1 <= sites <= 2^31-1 (got n = %lld, sites = %lld)", who, (long long)n,
                       (long long)sites);
        return FNN_E_ARG;
    }
    if (model < FNN_DIST_P || model > FNN_DIST_K2P) { fnn::set_error("%s: unknown distance model %d", who, model); return FNN_E_ARG; }
    if (!std::isnan(undef) && !(std::isfinite(undef) && undef >= 0.0)) {
        fnn::set_error("%s: undefined_value must be NaN (fail on an undefined pair) or finite and >= 0, got %g", who, undef);
        return FNN_E_ARG;
    }
    return FNN_OK;
}

namespace {

// v, m, s of one pair on the host, for the error message (sites: the replicate's columns, NULL = all)
void host_counts(const uint8_t* codes, int64_t L, const int32_t* sites, int64_t i, int64_t j, long long* v, long long* m, long long* s) {
    *v = *m = *s = 0;
    const uint8_t *x = codes + i * L, *y = codes + j * L;
    for (int64_t k = 0; k < L; ++k) {
        const int64_t col = sites ? sites[k] : k;
        if (x[col] < 4 && y[col] < 4) {
            ++*v;
            if (x[col] != y[col]) { ++*m; if ((x[col] ^ y[col]) == 2) ++*s; }
        }
    }
}

}  // namespace

int DistJob::upload(cudaStream_t stream_, int sms_, const uint8_t* codes_, int64_t n_, int64_t L_, bool resample, DistTimes* tm) {
    stream = stream_; sms = sms_; codes = codes_; n = n_; L = L_;
    const int64_t W = (L + 63) / 64, stages = (W + BK - 1) / BK, np = (n + TM - 1) / TM * TM;
    const size_t plane_bytes = sizeof(unsigned long long) * PLANES * (size_t)(stages * BK) * (size_t)np;
    FNN_CUDA(scratch.alloc((void**)&d_codes, (size_t)n * (size_t)L));
    FNN_CUDA(scratch.alloc((void**)&d_planes, plane_bytes));
    FNN_CUDA(scratch.alloc((void**)&d_flags, 2 * sizeof(unsigned long long)));
    if (resample) FNN_CUDA(scratch.alloc((void**)&d_sites, sizeof(int32_t) * (size_t)L));
    // tail words and padding taxa: ok = 0.  k_pack never writes them, so this holds for every later pack.
    FNN_CUDA(cudaMemsetAsync(d_planes, 0, plane_bytes, stream));
    DevEvent e0, e1;
    FNN_CUDA(e0.create()); FNN_CUDA(e1.create());
    FNN_CUDA(cudaEventRecord(e0, stream));
    FNN_CUDA(cudaMemcpyAsync(d_codes, codes, (size_t)n * (size_t)L, cudaMemcpyHostToDevice, stream));
    FNN_CUDA(cudaEventRecord(e1, stream));
    FNN_CUDA(cudaStreamSynchronize(stream));
    if (tm) cudaEventElapsedTime(&tm->upload_ms, e0, e1);
    return FNN_OK;
}

int DistJob::run(const char* who, const char* where, int32_t model, double undef, const int32_t* sites, double* dD, int64_t ld,
                 DistTimes* tm) {
    const int64_t W = (L + 63) / 64, stages = (W + BK - 1) / BK, np = (n + TM - 1) / TM * TM, nt = np / TM;
    if (sites && !d_sites) { fnn::set_error("%s: no site list buffer", who); return FNN_E_STATE; }
    const unsigned long long init[2] = {~0ull, 0ull};   // [0] = first undefined pair key, [1] = bad-code flag
    FNN_CUDA(cudaMemcpyAsync(d_flags, init, sizeof(init), cudaMemcpyHostToDevice, stream));
    if (sites) FNN_CUDA(cudaMemcpyAsync(d_sites, sites, sizeof(int32_t) * (size_t)L, cudaMemcpyHostToDevice, stream));
    DevEvent e1, e2, e3;
    FNN_CUDA(e1.create()); FNN_CUDA(e2.create()); FNN_CUDA(e3.create());
    FNN_CUDA(cudaEventRecord(e1, stream));
    const int64_t units = n * W;
    const int pack_grid = (int)std::min<int64_t>((units + 7) / 8, (int64_t)sms * 64);
    k_pack<<<pack_grid, 256, 0, stream>>>(d_codes, n, L, W, np, sites ? d_sites : nullptr, d_planes, (int*)(d_flags + 1));
    FNN_CUDA(cudaGetLastError());
    FNN_CUDA(cudaEventRecord(e2, stream));
    const int64_t tiles = nt * (nt + 1) / 2;
    const int fail = std::isnan(undef) ? 1 : 0;
    const double sub = fail ? 0.0 : undef;
    if (model == FNN_DIST_P) k_pairs<FNN_DIST_P><<<(unsigned)tiles, THREADS, 0, stream>>>(d_planes, np, stages, (int)n, dD, ld, sub, fail, d_flags);
    else if (model == FNN_DIST_JC69) k_pairs<FNN_DIST_JC69><<<(unsigned)tiles, THREADS, 0, stream>>>(d_planes, np, stages, (int)n, dD, ld, sub, fail, d_flags);
    else k_pairs<FNN_DIST_K2P><<<(unsigned)tiles, THREADS, 0, stream>>>(d_planes, np, stages, (int)n, dD, ld, sub, fail, d_flags);
    FNN_CUDA(cudaGetLastError());
    FNN_CUDA(cudaEventRecord(e3, stream));
    unsigned long long flags[2];
    FNN_CUDA(cudaMemcpyAsync(flags, d_flags, sizeof(flags), cudaMemcpyDeviceToHost, stream));
    FNN_CUDA(cudaStreamSynchronize(stream));
    if (tm) {
        cudaEventElapsedTime(&tm->pack_ms, e1, e2);
        cudaEventElapsedTime(&tm->pairs_ms, e2, e3);
    }
    if (flags[1]) { fnn::set_error("%s: a code is outside 0..4 (A C G T, 4 = missing)", who); return FNN_E_ARG; }
    if (flags[0] != ~0ull) {
        const int64_t i = (int64_t)(flags[0] / (unsigned long long)n), j = (int64_t)(flags[0] % (unsigned long long)n);
        long long v, m, s;
        host_counts(codes, L, sites, i, j, &v, &m, &s);
        fnn::set_error("%s: %sthe %s distance of pair (%lld, %lld) is undefined: v = %lld comparable sites, m = %lld differences, "
                       "s = %lld transitions; pass a finite undefined_value >= 0 to substitute it", who, where, model_name(model),
                       (long long)i, (long long)j, v, m, s);
        return FNN_E_ARG;
    }
    return FNN_OK;
}

extern "C" int fnn_ctx_load_alignment(fnn_ctx* c, const uint8_t* codes, int64_t sites, int32_t model, double undefined_value) {
    if (!c) { fnn::set_error("fnn_ctx_load_alignment: null context"); return FNN_E_ARG; }
    const int64_t n = fnn_ctx_n_(c);
    int rc = fnn_dist_check_args_("fnn_ctx_load_alignment", codes, n, sites, model, undefined_value);
    if (rc) return rc;
    FNN_CUDA(cudaSetDevice(fnn_ctx_device_(c)));
    double* dD;
    int64_t ld;
    fnn_ctx_matrix_ptr(c, &dD, &ld);
    fnn_ctx_mark_unloaded_(c);   // the matrix is overwritten; it counts as loaded only once the call succeeds
    DistTimes tm;
    DistJob job;
    rc = job.upload(fnn_ctx_stream_(c), fnn_ctx_sms_(c), codes, n, sites, false, &tm);
    if (!rc) rc = job.run("fnn_ctx_load_alignment", "", model, undefined_value, nullptr, dD, ld, &tm);
    if (rc) return rc;
    fnn_stats* st = fnn_ctx_stats_(c);
    st->h2d_ms = tm.upload_ms;
    st->reserved[6] = tm.pack_ms;
    st->reserved[7] = tm.pairs_ms;
    fnn_ctx_mark_loaded_(c);
    return FNN_OK;
}

extern "C" int fnn_distances(const fnn_opts* o, const uint8_t* codes, int64_t n, int64_t sites, int32_t model, double undefined_value,
                             double* D_out) {
    int rc = fnn_dist_check_args_("fnn_distances", codes, n, sites, model, undefined_value);
    if (rc) return rc;
    if (!D_out) { fnn::set_error("fnn_distances: null D_out"); return FNN_E_ARG; }
    int cnt = 0;
    if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt <= 0) {
        cudaGetLastError();
        fnn::set_error("no CUDA device available (libfastnn has no CPU fallback)");
        return FNN_E_NODEVICE;
    }
    const int dev = o ? o->device : 0;
    if (dev < 0 || dev >= cnt) { fnn::set_error("device %d out of range (%d devices)", dev, cnt); return FNN_E_ARG; }
    FNN_CUDA(cudaSetDevice(dev));
    int sms = 0;
    FNN_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    cudaStream_t stream;
    FNN_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    struct StreamGuard { cudaStream_t s; ~StreamGuard() { cudaStreamDestroy(s); } } guard{stream};
    double* dD = nullptr;
    DevScratch scratch;
    FNN_CUDA(scratch.alloc((void**)&dD, sizeof(double) * (size_t)n * (size_t)n));
    DistJob job;
    rc = job.upload(stream, sms, codes, n, sites, false, nullptr);
    if (!rc) rc = job.run("fnn_distances", "", model, undefined_value, nullptr, dD, n, nullptr);
    if (rc) return rc;
    FNN_CUDA(cudaMemcpyAsync(D_out, dD, sizeof(double) * (size_t)n * (size_t)n, cudaMemcpyDeviceToHost, stream));
    FNN_CUDA(cudaStreamSynchronize(stream));
    return FNN_OK;
}
