// fnn_boot.cu — bootstrap support of a network's splits (fnn_bootstrap, DESIGN.md §4.5).  Every replicate stays on the
// device: the alignment's codes are uploaded once, a replicate's bit-planes are packed through its sorted column draws
// (k_pack of csrc/fnn_dist.cu), the pair kernel writes the context's matrix, and the chain of fnn_network (ordering, split
// weights, compaction) leaves the replicate's kept splits on the device, where k_support matches them against the original
// network's kept splits:
//
//   Every original split {O[i+1..j]} (0 <= i < j <= n-1) excludes taxon O[n].  For a replicate split T = {O_r[a+1..b]} let U
//   be T, or its complement O_r[1..a] u O_r[b+1..n] when O[n] is in T: U is the side of the bipartition without O[n].  With
//   pos[t] the position of taxon t in O, lo = min pos(U) and hi = max pos(U), U is an original split iff hi - lo + 1 = |U|
//   (its positions are contiguous) and (lo - 1, hi) is among the original kept (i, j).  O[n] is in T iff max pos(T) = n.
//
//   k_support_table  one block: the sparse tables of range minima / maxima of pos(O_r[p + 1]), p = 0..n-1
//   k_support        one thread per kept replicate split: two or four table lookups, a binary search in the original kept
//                    packed indices (increasing), atomicAdd on support[k]
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>
#include "fastnn.h"
#include "fnn_common.h"
#include "fnn_relaxed_sm.h"

namespace {

constexpr int LEVELS_MAX = 16;   // 2^15 > 20 000 positions
constexpr int TABLE_THREADS = 1024;
constexpr int SUPPORT_THREADS = 256;

__host__ __device__ inline int64_t row_start(int64_t n, int64_t i) { return i * (2 * n - i - 1) / 2; }

// level k holds the minimum (maximum) of entries p .. p + 2^k - 1 at [k * n + p]
__global__ void __launch_bounds__(TABLE_THREADS) k_support_table(const int* __restrict__ ord_r, const int* __restrict__ pos, int n,
                                                                 int levels, int* __restrict__ tmin, int* __restrict__ tmax) {
    for (int p = threadIdx.x; p < n; p += TABLE_THREADS) tmin[p] = tmax[p] = pos[ord_r[p + 1]];
    __syncthreads();
    for (int k = 1; k < levels; ++k) {
        const int half = 1 << (k - 1), len = n - (1 << k) + 1;
        const int *pmin = tmin + (int64_t)(k - 1) * n, *pmax = tmax + (int64_t)(k - 1) * n;
        for (int p = threadIdx.x; p < len; p += TABLE_THREADS) {
            tmin[(int64_t)k * n + p] = min(pmin[p], pmin[p + half]);
            tmax[(int64_t)k * n + p] = max(pmax[p], pmax[p + half]);
        }
        __syncthreads();
    }
}

// min and max of entries l..r (inclusive, l <= r)
__device__ __forceinline__ void range_minmax(const int* __restrict__ tmin, const int* __restrict__ tmax, int n, int l, int r, int* mn,
                                             int* mx) {
    const int k = 31 - __clz(r - l + 1);
    const int64_t o = (int64_t)k * n;
    *mn = min(tmin[o + l], tmin[o + r - (1 << k) + 1]);
    *mx = max(tmax[o + l], tmax[o + r - (1 << k) + 1]);
}

__global__ void __launch_bounds__(SUPPORT_THREADS) k_support(const int* __restrict__ kept_r, int64_t kept, int n, const int* __restrict__ tmin,
                                                             const int* __restrict__ tmax, const int* __restrict__ orig_idx, int64_t orig_kept,
                                                             int* __restrict__ support) {
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < kept; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t idx = kept_r[q];
        int64_t a = 0, top = n - 2;   // the row a of the packed index: largest a with row_start(n, a) <= idx
        while (a < top) {
            const int64_t mid = (a + top + 1) >> 1;
            if (row_start(n, mid) <= idx) a = mid; else top = mid - 1;
        }
        const int64_t b = idx - row_start(n, a) + a + 1;
        // T = O_r[a+1 .. b] = table entries a .. b-1
        int lo, hi;
        range_minmax(tmin, tmax, n, (int)a, (int)b - 1, &lo, &hi);
        int64_t size = b - a;
        if (hi == n) {   // O[n] is in T: U is the complement, entries 0 .. a-1 and b .. n-1 (b <= n-1, so the second is never empty)
            size = n - size;
            range_minmax(tmin, tmax, n, (int)b, n - 1, &lo, &hi);
            if (a > 0) {
                int l2, h2;
                range_minmax(tmin, tmax, n, 0, (int)a - 1, &l2, &h2);
                lo = min(lo, l2);
                hi = max(hi, h2);
            }
        }
        if ((int64_t)(hi - lo + 1) != size) continue;
        const long long key = row_start(n, lo - 1) + (hi - lo);   // packed index of (i, j) = (lo - 1, hi)
        int64_t l = 0, r = orig_kept;
        while (l < r) {
            const int64_t mid = (l + r) >> 1;
            if ((long long)orig_idx[mid] < key) l = mid + 1; else r = mid;
        }
        if (l < orig_kept && (long long)orig_idx[l] == key) atomicAdd(&support[l], 1);
    }
}

// device buffers of the matching, for the whole call
struct SupportWork {
    int64_t n = 0;
    int levels = 0;
    int *pos = nullptr, *ord_r = nullptr, *tmin = nullptr, *tmax = nullptr, *orig_idx = nullptr, *support = nullptr;
    int64_t orig_kept = 0;
    DevScratch scratch;
};

// the original network: the position of every taxon in O and its kept packed indices, copied off the chain's workspace
int support_setup(SupportWork& s, cudaStream_t st, int64_t n, const int32_t* ordering, const int* d_kept_idx, int64_t kept) {
    s.n = n;
    s.levels = 1;
    while ((int64_t)1 << s.levels <= n) ++s.levels;
    std::vector<int> pos((size_t)n + 1, 0);
    for (int64_t p = 1; p <= n; ++p) pos[(size_t)ordering[p]] = (int)p;
    FNN_CUDA(s.scratch.alloc((void**)&s.pos, sizeof(int) * (size_t)(n + 1)));
    FNN_CUDA(s.scratch.alloc((void**)&s.ord_r, sizeof(int) * (size_t)(n + 1)));
    FNN_CUDA(s.scratch.alloc((void**)&s.tmin, sizeof(int) * (size_t)s.levels * (size_t)n));
    FNN_CUDA(s.scratch.alloc((void**)&s.tmax, sizeof(int) * (size_t)s.levels * (size_t)n));
    FNN_CUDA(s.scratch.alloc((void**)&s.orig_idx, sizeof(int) * (size_t)std::max<int64_t>(1, kept)));
    FNN_CUDA(s.scratch.alloc((void**)&s.support, sizeof(int) * (size_t)std::max<int64_t>(1, kept)));
    s.orig_kept = kept;
    FNN_CUDA(cudaMemcpyAsync(s.pos, pos.data(), sizeof(int) * (size_t)(n + 1), cudaMemcpyHostToDevice, st));
    if (kept > 0) FNN_CUDA(cudaMemcpyAsync(s.orig_idx, d_kept_idx, sizeof(int) * (size_t)kept, cudaMemcpyDeviceToDevice, st));
    FNN_CUDA(cudaMemsetAsync(s.support, 0, sizeof(int) * (size_t)std::max<int64_t>(1, kept), st));
    FNN_CUDA(cudaStreamSynchronize(st));   // pos lives on this stack frame's vector
    return FNN_OK;
}

// one replicate's kept splits (on the device, d_kept_idx) against the original's
int support_add(SupportWork& s, cudaStream_t st, const int32_t* ordering_r, const int* d_kept_idx, int64_t kept) {
    if (kept <= 0 || s.orig_kept <= 0) return FNN_OK;
    FNN_CUDA(cudaMemcpyAsync(s.ord_r, ordering_r, sizeof(int) * (size_t)(s.n + 1), cudaMemcpyHostToDevice, st));
    k_support_table<<<1, TABLE_THREADS, 0, st>>>(s.ord_r, s.pos, (int)s.n, s.levels, s.tmin, s.tmax);
    const int grid = (int)std::min<int64_t>((kept + SUPPORT_THREADS - 1) / SUPPORT_THREADS, 148 * 8);
    k_support<<<grid, SUPPORT_THREADS, 0, st>>>(d_kept_idx, kept, (int)s.n, s.tmin, s.tmax, s.orig_idx, s.orig_kept, s.support);
    FNN_CUDA(cudaGetLastError());
    return FNN_OK;
}

}  // namespace

extern "C" int fnn_bootstrap(const fnn_opts* o, const uint8_t* codes, int64_t n, int64_t sites, int32_t model, double undefined_value,
                             int32_t replicates, int64_t boot_seed, double cutoff, int32_t* ordering_out, int32_t* split_i,
                             int32_t* split_j, double* weight, int32_t* support, int64_t max_out, int64_t* n_out,
                             int32_t* replicate_orderings, int64_t* replicate_kept, double* times_out) {
    int rc = fnn_dist_check_args_("fnn_bootstrap", codes, n, sites, model, undefined_value);
    if (rc) return rc;
    if (n < 4 || n > 20000 || replicates < 1 || !ordering_out || !split_i || !split_j || !weight || !support || !n_out || max_out < 0) {
        fnn::set_error("fnn_bootstrap: bad arguments (4 <= n <= 20000, replicates >= 1, every output but the optional three given)");
        return FNN_E_ARG;
    }
    fnn_ctx* ctx = nullptr;
    rc = fnn_ctx_create(o, n, &ctx);
    if (rc) return rc;
    NetChain* w = nullptr;
    double acc[5] = {0, 0, 0, 0, 0};   // distances, ordering, split weights, matching (ms), CG iterations: replicates only
    rc = [&]() -> int {
        cudaStream_t cs = fnn_ctx_stream_(ctx);
        double* dD; int64_t ld;
        fnn_ctx_matrix_ptr(ctx, &dD, &ld);
        DistJob job;
        int r = job.upload(cs, fnn_ctx_sms_(ctx), codes, n, sites, true, nullptr);
        if (r) return r;
        r = fnn_chain_create_(o, n, &w);
        if (r) return r;
        // the original network: what fnn_network(fnn_distances(codes)) returns
        fnn_ctx_mark_unloaded_(ctx);
        r = job.run("fnn_bootstrap", "", model, undefined_value, nullptr, dD, ld, nullptr);
        if (r) return r;
        fnn_ctx_mark_loaded_(ctx);
        int64_t kept = 0;
        r = fnn_chain_run_(w, ctx, cutoff, ordering_out, &kept, nullptr);
        if (r) return r;
        *n_out = kept;
        if (kept > max_out) { fnn::set_error("fnn_bootstrap: %lld splits kept, room for %lld", (long long)kept, (long long)max_out); return FNN_E_ARG; }
        r = fnn_chain_copy_kept_(w, kept, split_i, split_j, weight);
        if (r) return r;
        cudaStream_t ws = fnn_chain_stream_(w);
        SupportWork sw;
        r = support_setup(sw, ws, n, ordering_out, fnn_chain_kept_idx_(w), kept);
        if (r) return r;
        // replicates: one java.util.Random(boot_seed) stream, L draws of nextInt(L) each, sorted by a counting sort
        unsigned long long rng = ((unsigned long long)boot_seed ^ 0x5DEECE66DULL) & ((1ULL << 48) - 1);
        std::vector<int32_t> count((size_t)sites), list((size_t)sites);
        std::vector<int32_t> ord_r((size_t)n + 1);
        DevEvent m0, m1;
        FNN_CUDA(m0.create()); FNN_CUDA(m1.create());
        char where[48];
        for (int32_t rep = 0; rep < replicates; ++rep) {
            std::fill(count.begin(), count.end(), 0);
            for (int64_t k = 0; k < sites; ++k) ++count[(size_t)relaxed::jr_next_int(rng, (int)sites)];
            for (int64_t col = 0, k = 0; col < sites; ++col)
                for (int32_t c = 0; c < count[(size_t)col]; ++c) list[(size_t)k++] = (int32_t)col;
            snprintf(where, sizeof(where), "replicate %d: ", rep);
            DistTimes dt;
            fnn_ctx_mark_unloaded_(ctx);
            r = job.run("fnn_bootstrap", where, model, undefined_value, list.data(), dD, ld, &dt);
            if (r) return r;
            fnn_ctx_mark_loaded_(ctx);
            int64_t kept_r = 0;
            ChainTimes ct;
            r = fnn_chain_run_(w, ctx, cutoff, ord_r.data(), &kept_r, &ct);
            if (r) return r;
            FNN_CUDA(cudaEventRecord(m0, ws));
            r = support_add(sw, ws, ord_r.data(), fnn_chain_kept_idx_(w), kept_r);
            if (r) return r;
            FNN_CUDA(cudaEventRecord(m1, ws));
            FNN_CUDA(cudaStreamSynchronize(ws));   // ord_r is reused and the kept indices are overwritten by the next replicate
            float mm = 0;
            cudaEventElapsedTime(&mm, m0, m1);
            acc[0] += (double)dt.pack_ms + (double)dt.pairs_ms;
            acc[1] += ct.order_ms;
            acc[2] += ct.csw_ms;
            acc[3] += mm;
            acc[4] += (double)ct.cg_iters;
            if (replicate_orderings) memcpy(replicate_orderings + (size_t)rep * (size_t)(n + 1), ord_r.data(), sizeof(int32_t) * (size_t)(n + 1));
            if (replicate_kept) replicate_kept[rep] = kept_r;
        }
        if (kept > 0) FNN_CUDA(cudaMemcpyAsync(support, sw.support, sizeof(int32_t) * (size_t)kept, cudaMemcpyDeviceToHost, ws));
        FNN_CUDA(cudaStreamSynchronize(ws));
        return FNN_OK;
    }();
    fnn_chain_destroy_(w);
    fnn_ctx_destroy(ctx);
    if (!rc && times_out) memcpy(times_out, acc, sizeof(acc));
    return rc;
}
