// fnn_csw.cu — seam B2: circular split weights (CircularSplitWeights.java) on the B200.
//
// Reference algorithm (kept): unconstrained closed form (CircularSplitWeights.java:247-271), then the
// active-set method with conjugate gradients on A^T A x = A^T d restricted to the free set
// (:359-557, :769-831), 60 % collapse (:282-330), min-ratio step (:438-460), most-negative
// active gradient release (:464-555).  W == 1 ("ols", :172-177, :213-236).
//
// What changes (B200-first): the two mat-vecs are not the reference's n-1 dependent wavefronts
// (:603-633, :643-731) but ONE primitive - the 2-D inclusive prefix sum P of the packed upper
// triangle (a warp-per-row scan, then a thread-per-column scan) - followed by O(1) gathers:
//     (Ab)(a,b)  = 2P(a-1,b-1) - P(a-1,a-1) + P(b-1,n-1) - P(a-1,n-1) - P(b-1,b-1)
//     (A^T d)(i,j) = (PRS[j] - PRS[i]) - 2 (G(j,j) - G(i,j)),  G = prefix2d(d), PRS = prefix of row sums
// Dot products use a fixed two-level tree.  Every summation order here is restated literally
// by the L1 oracle (oracle/csw_l1.cpp), so the active-set path - and therefore the weights - are
// bit-identical to it; the distance to the reference's own summation order (L0) is the
// algorithm's intrinsic noise floor (SURVEY F5) and is reported by the tests.
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <vector>
#include <algorithm>
#include <chrono>
#include "fastnn.h"
#include "fnn_common.h"
#include "fnn_exact_sum.cuh"

namespace {

struct Scalars {
    double rho, rho_old, e0sq, alpha, beta, dot;
    long long k, kmax, iters_total;
    int done;
    int pad;
};

__host__ __device__ inline int64_t row_start(int64_t n, int64_t i) { return i * (2 * n - i - 1) / 2; }
__host__ __device__ inline int64_t pidx(int64_t n, int64_t i, int64_t j) { return i * (2 * n - i - 3) / 2 + j - 1; }

// ---------------------------------------------------------------- prefix2d: row pass
// warp per row; blocks of 32 elements scanned Kogge-Stone, carry added sequentially
__global__ void k_rowscan(const double* __restrict__ v, double* __restrict__ Rw, double* __restrict__ RT, int n,
                          const int* done) {
    if (done && *done) return;
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    for (int64_t i = (int64_t)blockIdx.x * wpb + (threadIdx.x >> 5); i < n - 1; i += (int64_t)gridDim.x * wpb) {
        const int64_t rs = row_start(n, i);
        const int len = n - 1 - (int)i;
        double carry = 0.0;
        for (int blk = 0; blk < len; blk += 32) {
            double e = (blk + lane < len) ? v[rs + blk + lane] : 0.0;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const double t = __shfl_up_sync(0xffffffffu, e, off);
                if (lane >= off) e = e + t;
            }
            const double out = carry + e;
            if (blk + lane < len) Rw[rs + blk + lane] = out;
            carry = __shfl_sync(0xffffffffu, out, 31);
        }
        if (RT && lane == 0) RT[i] = carry;
    }
    if (RT && blockIdx.x == 0 && threadIdx.x == 0) RT[n - 1] = 0.0;
}

// ---------------------------------------------------------------- prefix2d: column pass (+ raw column sums)
// Blocked like the row pass: chunks of 32 rows are scanned top to bottom from zero (k_colscan_local), the chunk
// totals are accumulated sequentially per column (k_colscan_carry), and the carry is added to every entry
// (k_colscan_fix): P(i,j) = carry(chunk(i), j) + local(i, j).  Parallelism n * n/32 instead of n.
constexpr int COL_CHUNK = 32;

template <bool WITH_CT>
__global__ void k_colscan_local(const double* __restrict__ Rw, const double* __restrict__ v, double* __restrict__ P,
                                double* __restrict__ T, double* __restrict__ T2, int n, const int* done) {
    if (done && *done) return;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = blockIdx.y;
    if (j >= n) return;
    const int i0 = c * COL_CHUNK, i1 = min(i0 + COL_CHUNK, j);   // rows i < j
    double acc = 0.0, acc2 = 0.0;
    if (i0 < i1) {
        int64_t q = pidx(n, i0, j);
        for (int i = i0; i < i1; ++i) {
            acc = acc + Rw[q];
            P[q] = acc;
            if (WITH_CT) acc2 = acc2 + v[q];
            q += n - i - 2;
        }
    }
    T[(int64_t)c * n + j] = acc;
    if (WITH_CT) T2[(int64_t)c * n + j] = acc2;
}

template <bool WITH_CT>
__global__ void k_colscan_carry(double* __restrict__ T, const double* __restrict__ T2, double* __restrict__ CT, int n, int nchunks,
                                const int* done) {
    if (done && *done) return;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    double carry = 0.0, acc2 = 0.0;
    for (int c = 0; c < nchunks; ++c) {   // T[c][j] becomes the exclusive carry of chunk c
        const double t = T[(int64_t)c * n + j];
        T[(int64_t)c * n + j] = carry;
        carry = carry + t;
        if (WITH_CT) acc2 = acc2 + T2[(int64_t)c * n + j];
    }
    if (WITH_CT) CT[j] = acc2;
}

__global__ void k_colscan_fix(double* __restrict__ P, const double* __restrict__ T, int n, const int* done) {
    if (done && *done) return;
    const int i = blockIdx.y;
    if (i > n - 2) return;
    const double* carry = T + (int64_t)(i / COL_CHUNK) * n;
    const int64_t rs = row_start(n, i);
    for (int j = i + 1 + blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        const int64_t q = rs + (j - i - 1);
        P[q] = carry[j] + P[q];
    }
}

// PRS[a] = prefix over a' <= a of (RT[a'] + CT[a']): blocks of 32 scanned Kogge-Stone, carry added sequentially (the order of
// the row pass; a single dependent chain of n adds cost ~13 us at n = 800).  One warp.
__device__ __forceinline__ void prs_scan_warp(const double* RT, const double* CT, double* PRS, int n, int lane) {
    double carry = 0.0;
    for (int blk = 0; blk < n; blk += 32) {
        double e = (blk + lane < n) ? RT[blk + lane] + CT[blk + lane] : 0.0;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const double t = __shfl_up_sync(0xffffffffu, e, off);
            if (lane >= off) e = e + t;
        }
        const double out = carry + e;
        if (blk + lane < n) PRS[blk + lane] = out;
        carry = __shfl_sync(0xffffffffu, out, 31);
    }
}
__global__ void __launch_bounds__(32) k_prs(const double* RT, const double* CT, double* PRS, int n, const int* done) {
    if (done && *done) return;
    prs_scan_warp(RT, CT, PRS, n, threadIdx.x);
}

// ---------------------------------------------------------------- fixed reduction tree (level 1 inside producers)
// 256 threads own 4 consecutive values each: ((e0+e1)+e2)+e3, xor-butterfly in the warp, 8 warp totals added in order.
__device__ __forceinline__ double block_tree_1024(double s, double* sh8) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s = s + __shfl_xor_sync(0xffffffffu, s, off);
    if ((threadIdx.x & 31) == 0) sh8[threadIdx.x >> 5] = s;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0) {
        t = sh8[0];
        for (int w = 1; w < 8; ++w) t = t + sh8[w];
    }
    return t;   // valid in thread 0
}

enum Epilogue { EP_NONE = 0, EP_ALPHA = 1, EP_RHO_STEP = 2, EP_RHO_INIT = 3, EP_E0 = 4 };

__device__ void run_epilogue(int ep, double val, Scalars* sc) {
    if (ep == EP_ALPHA) { sc->dot = val; sc->alpha = sc->rho / val; }
    else if (ep == EP_RHO_STEP || ep == EP_RHO_INIT) {
        if (ep == EP_RHO_STEP) { sc->rho_old = sc->rho; sc->iters_total += 1; }
        else sc->rho_old = 0.0;
        sc->rho = val;
        // loop test of CircularSplitWeights.java:796: while ((rho > e_0*e_0) && (k < kmax))
        if ((val > sc->e0sq) && (sc->k < sc->kmax)) { sc->k += 1; if (sc->k > 1) sc->beta = val / sc->rho_old; }
        else sc->done = 1;
    } else if (ep == EP_E0) {
        const double e0 = 1e-8 * sqrt(val);   // CG_EPSILON * sqrt(norm(b)), :794
        sc->e0sq = e0 * e0;
    } else sc->dot = val;
}

// level >= 2: one block per 1024 partials; the last level (gridDim.x == 1) runs the epilogue
__global__ void __launch_bounds__(256) k_tree_level(const double* __restrict__ in, int64_t len, double* __restrict__ out,
                                                    int ep, Scalars* sc, int gated) {
    if (gated && sc->done) return;
    __shared__ double sh8[8];
    const int64_t base = (int64_t)blockIdx.x * 1024 + 4 * threadIdx.x;
    double e[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) e[q] = (base + q < len) ? in[base + q] : 0.0;
    const double s = ((e[0] + e[1]) + e[2]) + e[3];
    const double t = block_tree_1024(s, sh8);
    if (threadIdx.x == 0) {
        if (gridDim.x == 1) run_epilogue(ep, t, sc);
        else out[blockIdx.x] = t;
    }
}

// ---------------------------------------------------------------- Ab combine: d(a,b) from P
__global__ void k_ab_combine(const double* __restrict__ P, double* __restrict__ d, int n, const int* done) {
    if (done && *done) return;
    const int a = blockIdx.y;
    if (a >= n - 1) return;
    const double Pda = (a - 1 >= 1) ? P[pidx(n, a - 2, a - 1)] : 0.0;                 // P(a-1,a-1)
    const double Prowa = (a >= 1) ? P[pidx(n, a - 1, n - 1)] : 0.0;                    // P(a-1,n-1)
    for (int b = a + 1 + blockIdx.x * blockDim.x + threadIdx.x; b < n; b += gridDim.x * blockDim.x) {
        const double P1 = (a >= 1) ? P[pidx(n, a - 1, b - 1)] : 0.0;                   // P(a-1,b-1)
        const double Prowb = P[pidx(n, b - 1, n - 1)];                                  // P(b-1,n-1), b-1 <= n-2
        const double Pdb = (b - 1 >= 1) ? P[pidx(n, b - 2, b - 1)] : 0.0;              // P(b-1,b-1)
        double t = 2.0 * P1;
        t = t - Pda;
        t = t + Prowb;
        t = t - Prowa;
        t = t - Pdb;
        d[pidx(n, a, b)] = t;
    }
}

// ---------------------------------------------------------------- A^T d combine (+ optional mask and fused dot partials)
// MODE 0: out = p ; MODE 1: out = active ? 0 : p, partial[b] = tree(pvec * out) over this block's 1024 entries
template <int MODE>
__global__ void __launch_bounds__(256) k_atx_combine(const double* __restrict__ G, const double* __restrict__ PRS,
                                                     double* __restrict__ out, int n, int64_t npairs,
                                                     const unsigned char* __restrict__ active, const double* __restrict__ pvec,
                                                     double* __restrict__ partial, const int* done) {
    if (done && *done) return;
    __shared__ double sh8[8];
    const int64_t base = (int64_t)blockIdx.x * 1024 + 4 * threadIdx.x;
    double prod[4] = {0.0, 0.0, 0.0, 0.0};
    if (base < npairs) {
        // decode (i, j) of `base`, then walk
        int64_t i = (int64_t)(((2.0 * n - 1.0) - sqrt((2.0 * n - 1.0) * (2.0 * n - 1.0) - 8.0 * (double)base)) * 0.5);
        while (i > 0 && row_start(n, i) > base) --i;
        while (row_start(n, i + 1) <= base) ++i;
        int64_t j = base - row_start(n, i) + i + 1;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int64_t k = base + q;
            if (k < npairs) {
                const double u = PRS[j] - PRS[i];
                const double w = G[pidx(n, j - 1, j)] - G[k];      // G(j,j) - G(i,j); equal operands when i == j-1
                double pv = u - 2.0 * w;
                if (MODE == 1) {
                    if (active[k]) pv = 0.0;
                    prod[q] = pvec[k] * pv;
                }
                out[k] = pv;
                if (++j == n) { ++i; j = i + 1; }
            }
        }
    }
    if (MODE == 1) {
        const double s = ((prod[0] + prod[1]) + prod[2]) + prod[3];
        const double t = block_tree_1024(s, sh8);
        if (threadIdx.x == 0) partial[blockIdx.x] = t;
    }
}

// ---------------------------------------------------------------- unconstrained closed form (:247-271), one thread per entry
__global__ void k_unconstrained(const double* __restrict__ d, double* __restrict__ x, int n) {
    const int i = blockIdx.y;
    if (i > n - 2) return;
    const int64_t rs = row_start(n, i);
    for (int j = i + 1 + blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        const int64_t index = rs + (j - i - 1);
        double v;
        if (i == n - 2) v = (d[index] + d[n - 2] - d[n - 3]) / 2.0;                                  // last entry (:270)
        else if (j == i + 1) v = (d[index] + d[index + (n - i - 2) + 1] - d[index + 1]) / 2.0;       // :250
        else if (j <= n - 2) v = (d[index] + d[index + (n - i - 2) + 1] - d[index + 1] - d[index + (n - i - 2)]) / 2.0;  // :253
        else if (i == 0) v = (d[0] + d[n - 2] - d[2 * n - 4]) / 2.0;                                 // :257
        else v = (d[index] + d[i] - d[i - 1] - d[index + (n - i - 2)]) / 2.0;                        // :259
        x[index] = v;
    }
}

// ---------------------------------------------------------------- CG vector kernels
// r = active ? 0 : b - r ; partial = tree(r*r)
__global__ void __launch_bounds__(256) k_residual_init(double* __restrict__ r, const double* __restrict__ b,
                                                       const unsigned char* __restrict__ active, int64_t len,
                                                       double* __restrict__ partial) {
    __shared__ double sh8[8];
    const int64_t base = (int64_t)blockIdx.x * 1024 + 4 * threadIdx.x;
    double e[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int q = 0; q < 4; ++q)
        if (base + q < len) {
            const double v = active[base + q] ? 0.0 : b[base + q] - r[base + q];
            r[base + q] = v;
            e[q] = v * v;
        }
    const double t = block_tree_1024(((e[0] + e[1]) + e[2]) + e[3], sh8);
    if (threadIdx.x == 0) partial[blockIdx.x] = t;
}
__global__ void __launch_bounds__(256) k_square_partials(const double* __restrict__ v, int64_t len, double* __restrict__ partial) {
    __shared__ double sh8[8];
    const int64_t base = (int64_t)blockIdx.x * 1024 + 4 * threadIdx.x;
    double e[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int q = 0; q < 4; ++q)
        if (base + q < len) e[q] = v[base + q] * v[base + q];
    const double t = block_tree_1024(((e[0] + e[1]) + e[2]) + e[3], sh8);
    if (threadIdx.x == 0) partial[blockIdx.x] = t;
}
// p = (k == 1) ? r : r + beta * p      (:799-806)
__global__ void k_pupdate(double* __restrict__ p, const double* __restrict__ r, int64_t len, const Scalars* sc) {
    if (sc->done) return;
    const bool first = sc->k == 1;
    const double beta = sc->beta;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x)
        p[i] = first ? r[i] : r[i] + beta * p[i];
}
// x += alpha p ; r -= alpha w ; partial = tree(r*r)     (:822-828)
__global__ void __launch_bounds__(256) k_xr_update(double* __restrict__ x, double* __restrict__ r, const double* __restrict__ p,
                                                   const double* __restrict__ w, int64_t len, const Scalars* sc,
                                                   double* __restrict__ partial) {
    if (sc->done) return;
    __shared__ double sh8[8];
    const double alpha = sc->alpha;
    const int64_t base = (int64_t)blockIdx.x * 1024 + 4 * threadIdx.x;
    double e[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int q = 0; q < 4; ++q)
        if (base + q < len) {
            x[base + q] = x[base + q] + alpha * p[base + q];
            const double rv = r[base + q] - alpha * w[base + q];
            r[base + q] = rv;
            e[q] = rv * rv;
        }
    const double t = block_tree_1024(((e[0] + e[1]) + e[2]) + e[3], sh8);
    if (threadIdx.x == 0) partial[blockIdx.x] = t;
}

// ---------------------------------------------------------------- active-set helpers (hand-written: no library calls)
// State of the selection primitives, one per solver, in device memory.
struct SelState {
    unsigned long long prefix;    // radix select: digits of the k-th smallest key fixed so far
    long long k;                  // rank still to be located inside the current bucket (0-based)
    long long less;               // negatives strictly below the cutoff
    long long num_neg, nkept, ties, slots;
    double cutoff;
    unsigned int ticket, pad;
    unsigned int hist[256];
    long long flag_total;         // flag scan: number of set flags
    double ml_v; long long ml_i;  // min-loc result
};
constexpr int SEL_THREADS = 256;

// worstIndices (:282-330), step 1: count the negatives; the last block derives nkept = ceil(propKept * numNeg) (:309)
__global__ void __launch_bounds__(SEL_THREADS) k_sel_count_neg(const double* __restrict__ x, int64_t len, SelState* sel) {
    __shared__ long long wsum[SEL_THREADS / 32];
    long long cnt = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x) cnt += x[i] < 0.0;
    for (int off = 16; off > 0; off >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long t = 0;
        for (int w = 0; w < SEL_THREADS / 32; ++w) t += wsum[w];
        if (t) atomicAdd((unsigned long long*)&sel->num_neg, (unsigned long long)t);
        __threadfence();
        if (atomicAdd(&sel->ticket, 1u) == gridDim.x - 1) {
            __threadfence();
            const long long nn = *(volatile long long*)&sel->num_neg;
            const long long nkept = (long long)ceil(0.6 * (double)nn);
            sel->nkept = nkept; sel->k = nkept - 1; sel->prefix = 0; sel->less = 0; sel->ties = 0; sel->slots = 0;
            sel->ticket = 0;
        }
    }
}
// step 2: the cutoff = the nkept-th smallest negative (:310), by an exact 8 x 8-bit radix select instead of a full sort.
// For negative doubles, ascending value = ascending ~bits.  Pass p histograms digit p (from the top) of the keys that
// agree with the digits fixed so far; the last block picks the bucket holding rank k.
__global__ void __launch_bounds__(SEL_THREADS) k_sel_radix_pass(const double* __restrict__ x, int64_t len, SelState* sel, int pass) {
    if (sel->num_neg == 0) return;
    __shared__ unsigned int h[256];
    h[threadIdx.x] = 0;   // SEL_THREADS == 256
    __syncthreads();
    const int shift = 56 - 8 * pass;
    const unsigned long long prefix = sel->prefix;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x) {
        const double v = x[i];
        if (v < 0.0) {
            const unsigned long long key = ~(unsigned long long)__double_as_longlong(v);
            if (pass == 0 || (key >> (shift + 8)) == (prefix >> (shift + 8))) atomicAdd(&h[(key >> shift) & 255], 1u);
        }
    }
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(&sel->hist[threadIdx.x], h[threadIdx.x]);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(&sel->ticket, 1u) == gridDim.x - 1) {
        __threadfence();
        volatile unsigned int* gh = sel->hist;
        long long k = sel->k, less = sel->less;
        int b = 0;
        for (; b < 255; ++b) {
            const long long cb = gh[b];
            if (k < cb) break;
            k -= cb; less += cb;
        }
        sel->prefix = prefix | ((unsigned long long)b << shift);
        sel->k = k; sel->less = less;
        if (pass == 7) {
            sel->ties = gh[b];                                         // entries equal to the cutoff
            sel->cutoff = __longlong_as_double((long long)~sel->prefix);
            sel->slots = sel->nkept - less;                            // result slots left for ties (filled from the back, :321-327)
        }
        for (int q = 0; q < 256; ++q) gh[q] = 0;
        sel->ticket = 0;
    }
}
// step 3 (:314-328 + the contraction :422-431): x < cutoff -> contract; x == cutoff -> the EARLIEST ties fill the remaining
// slots.  When every tie fits (the common case: the cutoff value is unique) they are contracted here; otherwise they are
// flagged and ranked by the flag scan below.
__global__ void k_sel_mark(double* x, unsigned char* active, int64_t len, const SelState* sel, int* tie_flag) {
    if (sel->num_neg == 0) return;
    const double cutoff = sel->cutoff;
    const bool rank_ties = sel->ties > sel->slots;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x) {
        const double v = x[i];
        int f = 0;
        if (v < cutoff) { x[i] = 0.0; active[i] = 1; }
        else if (v == cutoff) {
            if (rank_ties) f = 1;
            else { x[i] = 0.0; active[i] = 1; }
        }
        tie_flag[i] = f;
    }
}
__global__ void k_sel_mark_ties(double* x, unsigned char* active, int64_t len, const SelState* sel, const int* tie_flag, const int* local_rank,
                                const long long* block_excl) {
    if (sel->num_neg == 0 || sel->ties <= sel->slots) return;
    const long long slots = sel->slots;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x)
        if (tie_flag[i] && block_excl[i >> 10] + local_rank[i] < slots) { x[i] = 0.0; active[i] = 1; }
}

// ---- exclusive prefix count of 0/1 flags in index order: rank(i) = block_excl[i / 1024] + local_rank[i]
__global__ void __launch_bounds__(1024) k_flag_local(const int* __restrict__ flag, int64_t len, int* __restrict__ local_rank,
                                                     long long* __restrict__ block_sum, const SelState* gate_ties) {
    if (gate_ties && (gate_ties->num_neg == 0 || gate_ties->ties <= gate_ties->slots)) return;
    __shared__ int wtot[32];
    const int64_t i = (int64_t)blockIdx.x * 1024 + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int f = (i < len) ? flag[i] : 0;
    const unsigned bal = __ballot_sync(0xffffffffu, f != 0);
    const int within = __popc(bal & ((1u << lane) - 1u));
    if (lane == 0) wtot[warp] = __popc(bal);
    __syncthreads();
    if (warp == 0) {
        int v = wtot[lane];
        const int own = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) { const int t = __shfl_up_sync(0xffffffffu, v, off); if (lane >= off) v += t; }
        wtot[lane] = v - own;
        if (lane == 31) block_sum[blockIdx.x] = v;
    }
    __syncthreads();
    if (i < len) local_rank[i] = wtot[warp] + within;
}
__global__ void __launch_bounds__(1024) k_flag_blockscan(long long* block_sum, int64_t nblk, SelState* sel, const SelState* gate_ties) {
    if (gate_ties && (gate_ties->num_neg == 0 || gate_ties->ties <= gate_ties->slots)) return;
    __shared__ long long wtot[32];
    __shared__ long long carry_s;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int64_t b0 = 0; b0 < nblk; b0 += 1024) {
        const int64_t b = b0 + threadIdx.x;
        long long v = (b < nblk) ? block_sum[b] : 0;
        const long long own = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) { const long long t = __shfl_up_sync(0xffffffffu, v, off); if (lane >= off) v += t; }
        if (lane == 31) wtot[warp] = v;
        __syncthreads();
        if (warp == 0) {
            long long w = wtot[lane];
            const long long wown = w;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) { const long long t = __shfl_up_sync(0xffffffffu, w, off); if (lane >= off) w += t; }
            wtot[lane] = w - wown;
        }
        __syncthreads();
        const long long carry = carry_s;
        if (b < nblk) block_sum[b] = carry + wtot[warp] + (v - own);   // exclusive
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = carry + wtot[31] + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) sel->flag_total = carry_s;
}

struct MinLoc { double v; long long i; };
struct MinLocOp {
    __device__ MinLoc operator()(const MinLoc& a, const MinLoc& b) const {
        if (a.i < 0) return b;
        if (b.i < 0) return a;
        return (b.v < a.v || (b.v == a.v && b.i < a.i)) ? b : a;   // first strict minimum in index order
    }
};
// (:438-448) xi = old_x / (old_x - x) over x < 0
struct RatioIn {
    const double* x; const double* old_x;
    __device__ MinLoc operator()(long long i) const {
        const double xv = x[i];
        if (xv < 0.0) return MinLoc{old_x[i] / (old_x[i] - xv), i};
        return MinLoc{0.0, -1};
    }
};
// (:464-479) r = (r - AtWd) * 2 ; min over active
__global__ void k_gradient(double* r, const double* AtWd, int64_t len) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x) {
        double v = r[i] - AtWd[i];
        r[i] = v * 2.0;
    }
}
struct GradIn {
    const double* r; const unsigned char* active;
    __device__ MinLoc operator()(long long i) const { return active[i] ? MinLoc{r[i], i} : MinLoc{0.0, -1}; }
};
// first strict minimum in index order over op(i), i < len (:438-448, :475-492, :369-374): grid-stride partials, then the last
// block to finish reduces them (MinLocOp is associative and commutative, so the result does not depend on the schedule)
template <typename InOp>
__global__ void __launch_bounds__(SEL_THREADS) k_minloc(InOp op, int64_t len, MinLoc* partials, SelState* sel) {
    __shared__ MinLoc wb[SEL_THREADS / 32];
    __shared__ bool amLast;
    MinLocOp red;
    MinLoc best{0.0, -1};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x) best = red(best, op(i));
    auto warp_reduce = [&](MinLoc v) {
        for (int off = 16; off > 0; off >>= 1) {
            MinLoc o;
            o.v = __shfl_xor_sync(0xffffffffu, v.v, off);
            o.i = __shfl_xor_sync(0xffffffffu, v.i, off);
            v = red(v, o);
        }
        return v;
    };
    best = warp_reduce(best);
    if ((threadIdx.x & 31) == 0) wb[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < SEL_THREADS / 32; ++w) best = red(best, wb[w]);
        partials[blockIdx.x] = best;
        __threadfence();
        amLast = (atomicAdd(&sel->ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (amLast) {
        __threadfence();
        MinLoc v{0.0, -1};
        for (int b = threadIdx.x; b < (int)gridDim.x; b += SEL_THREADS) {
            MinLoc pb;
            pb.v = __ldcg(&partials[b].v); pb.i = __ldcg(&partials[b].i);
            v = red(v, pb);
        }
        v = warp_reduce(v);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) wb[threadIdx.x >> 5] = v;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < SEL_THREADS / 32; ++w) v = red(v, wb[w]);
            sel->ml_v = v.v; sel->ml_i = v.i;
            sel->ticket = 0;
        }
    }
}

// (:452-455) old_x += min_xi * (x - old_x) on the free set
__global__ void k_oldx_step(double* old_x, const double* x, const unsigned char* active, int64_t len, double min_xi) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x)
        if (!active[i]) old_x[i] = old_x[i] + min_xi * (x[i] - old_x[i]);
}
__global__ void k_set_one(double* x, unsigned char* active, long long i, double xv, int av, int set_x) {
    if (threadIdx.x == 0 && blockIdx.x == 0) { if (set_x) x[i] = xv; active[i] = (unsigned char)av; }
}
__global__ void k_fill(double* v, int64_t len, double val) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x) v[i] = val;
}
// setupD with the rotated permutation (SURVEY F4): position 0 <-> ordering[n], position p <-> ordering[p]
__global__ void k_setup_d(const double* __restrict__ d_upper, const int* __restrict__ ordering, double* __restrict__ d_pos, int n) {
    const int i = blockIdx.y;
    if (i > n - 2) return;
    const int64_t ti = (i == 0 ? ordering[n] : ordering[i]) - 1;
    for (int j = i + 1 + blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        const int64_t tj = ordering[j] - 1;
        const int64_t a = ti < tj ? ti : tj, b = ti < tj ? tj : ti;
        d_pos[pidx(n, i, j)] = d_upper[a * (n - 1) - a * (a - 1) / 2 + b - (a + 1)];   // DistancesAndNames.upperIndex (:24-38)
    }
}


// ============================================================================ persistent CG loop (one launch per CG solve)
// The loop body of circularConjugateGrads (:797-829) is ~20 dependent launches in the graph path (~45-85 us per iteration
// regardless of n, 10^4-10^6 iterations per solve).  k_cg_persistent runs the WHOLE loop in one cooperative launch: the
// phases of an iteration are separated by grid barriers (one atomic + one acquire spin per CTA) instead of kernel
// boundaries.  Every scan, combine and reduction keeps the operand order of the per-phase kernels above, so the L1 oracle
// is the bit-exact check for both paths:
//   * the p update is fused into the row scan of A p; k_ab_combine is fused into the row scan of A^T y;
//   * k_colscan_fix is folded into its consumers: P stays chunk-local and every read adds its carry, `carry[j] + P[q]`,
//     exactly the operands and order of the in-place fix;
//   * PRS (one warp) and the upper levels of the two reduction trees are recomputed redundantly by every CTA, so alpha,
//     rho and the loop test need no broadcast and every CTA takes the same control decisions.
// 8 grid barriers per iteration.  Buffers written inside the kernel carry no const/__restrict__ (no ld.global.nc).
struct CgArgs {
    double *x, *r, *p, *w, *y, *Rw, *P, *RT, *CT, *T, *T2, *part1, *part2;
    const unsigned char* active;
    Scalars* sc;
    unsigned long long* bar;   // [0] arrivals (monotonic), [1] released generation
    int n, nchunks;
    long long np, nblk;
    long long max_iters;       // leave the kernel after this many iterations (0: run to the end): keeps single launches short
    unsigned long long* prof;  // optional (env FNN_CSW_PROF): ns per phase / barrier accumulated by CTA 0, [24]
};
constexpr int CGP_THREADS = 512;          // 128 registers per thread: the phases keep 16-24 independent loads in flight per thread
constexpr int CGP_Q = CGP_THREADS / 256;    // 256-thread groups, each owns one 1024-entry block of the reduction tree
constexpr int CGP_MAX_N = 12000;            // two n-vectors of doubles in shared memory (PRS / diagonal, row ends)

// Every phase is written as a few ROUNDS of independent loads (each thread first issues all loads of a small batch, then
// consumes them) instead of a chain of dependent ones: the solver is latency-bound at the sizes it is used at.  Batches are
// sized so that nothing spills: a spill store waits for its load and, issue being in order, serialises the whole batch
// (ncu, round 2: STL.64 with long-scoreboard stalls were the hot instructions of a 16-deep version).
// Cross-CTA data is read with ordinary (L1-cached) loads: the acquire of every grid barrier invalidates this SM's L1
// (SASS CCTL.IVALL), nothing is exchanged inside a phase, and per-thread runs of 4 consecutive doubles then cost one L2
// sector fetch instead of four (ld.global.cg made phases 8 and 10 L2-bandwidth-bound: x4 sector traffic).
__device__ __forceinline__ double ldg_cg(const double* p) { return *p; }

__device__ __forceinline__ void grid_barrier(unsigned long long* bar, unsigned long long nblocks, unsigned long long& gen) {
    __syncthreads();
    if (threadIdx.x == 0) {
        gen += 1;
        __threadfence();
        const unsigned long long prev = atomicAdd(&bar[0], 1ull);
        if (prev + 1 == nblocks * gen) {
            asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(&bar[1]), "l"(gen) : "memory");
        } else {
            unsigned long long g;   // relaxed polls (an acquire load invalidates L1 on every poll), one acquire fence at the end
            do { asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(g) : "l"(&bar[1]) : "memory"); } while (g < gen);
        }
        __threadfence();   // acquire side: orders the phase's loads after the release and drops this SM's stale L1 lines
    }
    __syncthreads();
}

// k_colscan_fix folded into the consumers: carry[j] + P[q]
__device__ __forceinline__ double fixed_P(const double* P, const double* T, int n, int i, int j) {
    return ldg_cg(T + (int64_t)(i / COL_CHUNK) * n + j) + ldg_cg(P + pidx(n, i, j));
}

// k_tree_level on one block of 1024 values read through `get`, by 256-thread group g of the CTA; result in the group's
// thread 0.  All threads call (two __syncthreads inside).
template <typename Get>
__device__ __forceinline__ double group_tree(Get get, long long base, long long len, int g, int t4, double (*sh8)[8]) {
    double e[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) e[q] = (base + 4 * t4 + q < len) ? get(base + 4 * t4 + q) : 0.0;
    double s = ((e[0] + e[1]) + e[2]) + e[3];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s = s + __shfl_xor_sync(0xffffffffu, s, off);
    if ((threadIdx.x & 31) == 0) sh8[g][(threadIdx.x >> 5) & 7] = s;
    __syncthreads();
    double t = 0.0;
    if (t4 == 0) {
        t = sh8[g][0];
        for (int w = 1; w < 8; ++w) t = t + sh8[g][w];
    }
    __syncthreads();
    return t;
}

// levels >= 2 of the fixed tree over part[0..nblk) (finish_tree), recomputed by every CTA; result to all threads.
// nblk <= 2^20: level 2 leaves at most 1024 values (in lv, shared), level 3 is the root.
__device__ double cgp_reduce(const double* part, long long nblk, double* lv, double (*sh8)[8], double* bval) {
    const int g = threadIdx.x >> 8, t4 = threadIdx.x & 255;
    const long long blocks2 = (nblk + 1023) / 1024;
    if (blocks2 == 1) {
        const double t = group_tree([&](long long k) { return ldg_cg(part + k); }, 0, g == 0 ? nblk : 0, g, t4, sh8);
        if (threadIdx.x == 0) *bval = t;
    } else {
        for (long long b0 = 0; b0 < blocks2; b0 += CGP_Q) {
            const long long vb = b0 + g;
            const double t = group_tree([&](long long k) { return ldg_cg(part + k); }, vb * 1024, vb < blocks2 ? nblk : 0, g, t4, sh8);
            if (t4 == 0 && vb < blocks2) lv[vb] = t;
        }
        __syncthreads();
        const double t = group_tree([&](long long k) { return lv[k]; }, 0, g == 0 ? blocks2 : 0, g, t4, sh8);
        if (threadIdx.x == 0) *bval = t;
    }
    __syncthreads();
    const double v = *bval;
    __syncthreads();
    return v;
}

// Kogge-Stone inclusive scan of one 32-block (no carry): the blocks of a row are independent up to here, so several of them
// are scanned back to back (their shuffle chains overlap) before the short sequential carry chain
//   out_b = carry_b + local_b,  carry_{b+1} = out_b[31]
// is applied - the same operands in the same order as scanning block after block, hence the same bits.
__device__ __forceinline__ double scan32_local(double e, int lane) {
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, e, off);
        if (lane >= off) e = e + t;
    }
    return e;
}
// chunk-local column scan of COL_CHUNK rows from zero (k_colscan_local): all loads of a half-chunk first, then the chain
template <bool WITH_CT>
__device__ __forceinline__ void colscan_local_thread(const double* Rw, const double* v, double* P, double* T, double* T2, int n, int c,
                                                     int j) {
    const int i0 = c * COL_CHUNK, i1 = min(i0 + COL_CHUNK, j);
    double acc = 0.0, acc2 = 0.0;
    int64_t q = (i0 < i1) ? pidx(n, i0, j) : 0;
    constexpr int B = WITH_CT ? 4 : 8;
    for (int h0 = i0; h0 < i1; h0 += B) {
        double rw[B], vv[WITH_CT ? B : 1];
        int64_t qq = q;
#pragma unroll
        for (int k = 0; k < B; ++k) {
            const int i = h0 + k;
            if (i < i1) {
                rw[k] = ldg_cg(Rw + qq);
                if (WITH_CT) vv[k] = ldg_cg(v + qq);
                qq += n - i - 2;
            }
        }
#pragma unroll
        for (int k = 0; k < B; ++k) {
            const int i = h0 + k;
            if (i < i1) {
                acc = acc + rw[k];
                P[q] = acc;
                if (WITH_CT) acc2 = acc2 + vv[k];
                q += n - i - 2;
            }
        }
    }
    T[(int64_t)c * n + j] = acc;
    if (WITH_CT) T2[(int64_t)c * n + j] = acc2;
}

// exclusive carries of the chunk totals of column j (k_colscan_carry), loads batched by 16
template <bool WITH_CT>
__device__ __forceinline__ void colscan_carry_thread(double* T, const double* T2, double* CT, int n, int nchunks, int j) {
    double carry = 0.0, acc2 = 0.0;
    constexpr int B = WITH_CT ? 4 : 8;
    for (int c0 = 0; c0 < nchunks; c0 += B) {
        double t[B], t2[WITH_CT ? B : 1];
#pragma unroll
        for (int k = 0; k < B; ++k)
            if (c0 + k < nchunks) {
                t[k] = ldg_cg(T + (int64_t)(c0 + k) * n + j);
                if (WITH_CT) t2[k] = ldg_cg(T2 + (int64_t)(c0 + k) * n + j);
            }
#pragma unroll
        for (int k = 0; k < B; ++k)
            if (c0 + k < nchunks) {
                T[(int64_t)(c0 + k) * n + j] = carry;
                carry = carry + t[k];
                if (WITH_CT) acc2 = acc2 + t2[k];
            }
    }
    if (WITH_CT) CT[j] = acc2;
}

template <bool PROF>
__global__ void __launch_bounds__(CGP_THREADS, 1) k_cg_persistent(CgArgs a) {
    extern __shared__ double dyn[];          // [0, n): PRS or the diagonal vector; [n, 2n): the row-end vector
    __shared__ double sh8[CGP_Q][8];
    __shared__ double lv[1024];
    __shared__ double bval;
    const int n = a.n, nchunks = a.nchunks;
    double* vecA = dyn;
    double* vecB = dyn + n;
    const long long np = a.np, nblk = a.nblk;
    const int tid = threadIdx.x, lane = tid & 31;
    // rows are dealt round-robin over the CTAs (row i -> CTA i % grid): the long rows (small i) bound the row-scan phases
    const int gwarp = (tid >> 5) * gridDim.x + blockIdx.x, nwarps = gridDim.x * (CGP_THREADS / 32);
    const long long gtid = (long long)blockIdx.x * CGP_THREADS + tid, gthreads = (long long)gridDim.x * CGP_THREADS;
    const int g = tid >> 8, t4 = tid & 255;
    const unsigned long long nblocks = gridDim.x;
    unsigned long long gen = 0;
    if (tid == 0) asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(gen) : "l"(&a.bar[1]) : "memory");   // resumed launches continue the count

    // loop-carried scalars, identical in every thread of every CTA
    double rho = a.sc->rho, rho_old = a.sc->rho_old, beta = a.sc->beta, alpha = a.sc->alpha, dot = a.sc->dot;
    const double e0sq = a.sc->e0sq;
    long long k = a.sc->k, iters_total = a.sc->iters_total;
    const long long kmax = a.sc->kmax;
    int done = a.sc->done;
    long long left = a.max_iters;
    constexpr int U = 4;   // 32-element blocks of a row in flight per warp
    unsigned long long tacc[PROF ? 20 : 1], tlast = 0;
    const bool prof = PROF && (a.prof != nullptr) && gtid == 0;
    if (PROF && prof) {
#pragma unroll
        for (int q = 0; q < 20; ++q) tacc[PROF ? q : 0] = 0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tlast));
    }
#define CG_MARK(slot)                                                        \
    if (PROF && prof) {                                                      \
        unsigned long long tn_;                                              \
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tn_));              \
        tacc[PROF ? slot : 0] += tn_ - tlast;                                \
        tlast = tn_;                                                         \
    }

    while (!done) {
        // ---- phase 1: p = (k == 1) ? r : r + beta p   (k_pupdate), row scan of p -> Rw   (k_rowscan, no RT)
        const bool first = (k == 1);
        for (int i = gwarp; i < n - 1; i += nwarps) {
            const int64_t rs = row_start(n, i);
            const int len = n - 1 - i;
            double carry = 0.0;
            for (int b0 = 0; b0 < len; b0 += 32 * U) {
                double rv[U], pv[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int idx = b0 + 32 * u + lane;
                    rv[u] = 0.0; pv[u] = 0.0;
                    if (idx < len) { rv[u] = ldg_cg(a.r + rs + idx); if (!first) pv[u] = ldg_cg(a.p + rs + idx); }
                }
                double loc[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {              // U independent block scans
                    const int idx = b0 + 32 * u + lane;
                    double e = 0.0;
                    if (idx < len) {
                        e = first ? rv[u] : rv[u] + beta * pv[u];
                        a.p[rs + idx] = e;
                    }
                    loc[u] = scan32_local(e, lane);
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {              // the carry chain
                    if (b0 + 32 * u < len) {
                        const int idx = b0 + 32 * u + lane;
                        const double out = carry + loc[u];
                        carry = __shfl_sync(0xffffffffu, out, 31);
                        if (idx < len) a.Rw[rs + idx] = out;
                    }
                }
            }
        }
        CG_MARK(0)
        grid_barrier(a.bar, nblocks, gen);
        CG_MARK(1)
        // ---- phase 2: k_colscan_local<false>
        for (long long idx = gtid; idx < (long long)nchunks * n; idx += gthreads)
            colscan_local_thread<false>(a.Rw, nullptr, a.P, a.T, a.T2, n, (int)(idx / n), (int)(idx % n));
        CG_MARK(2)
        grid_barrier(a.bar, nblocks, gen);
        CG_MARK(3)
        // ---- phase 3: k_colscan_carry<false>
        for (long long j = gtid; j < n; j += gthreads) colscan_carry_thread<false>(a.T, nullptr, nullptr, n, nchunks, (int)j);
        CG_MARK(4)
        grid_barrier(a.bar, nblocks, gen);
        CG_MARK(5)
        // ---- phase 4: y = A p from P (k_ab_combine, with the fix folded in), row scan of y -> Rw, RT   (k_rowscan)
        // the two n-vectors every entry needs, once per CTA: vecA[b] = P(b-1,b-1) = fixed P at (b-2, b-1), vecB[b] = P(b-1,n-1)
        for (int b = tid; b < n; b += CGP_THREADS) {
            vecA[b] = (b - 1 >= 1) ? fixed_P(a.P, a.T, n, b - 2, b - 1) : 0.0;
            vecB[b] = (b >= 1) ? fixed_P(a.P, a.T, n, b - 1, n - 1) : 0.0;
        }
        __syncthreads();
        for (int i = gwarp; i < n - 1; i += nwarps) {
            const int64_t rs = row_start(n, i);
            const int len = n - 1 - i;
            const double Pda = vecA[i];
            const double Prowa = vecB[i];
            const double* Trow = a.T + (int64_t)((i >= 1 ? i - 1 : 0) / COL_CHUNK) * n;
            const int64_t prow = (i >= 1) ? pidx(n, i - 1, 0) : 0;   // P(i-1, b-1) sits at prow + (b-1)
            double carry = 0.0;
            for (int b0 = 0; b0 < len; b0 += 32 * U) {
                double tc[U], pl[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int idx = b0 + 32 * u + lane;
                    tc[u] = 0.0; pl[u] = 0.0;
                    if (idx < len && i >= 1) {
                        const int b = i + 1 + idx;
                        tc[u] = ldg_cg(Trow + (b - 1));
                        pl[u] = ldg_cg(a.P + prow + (b - 1));
                    }
                }
                double loc[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {              // U independent block scans
                    const int idx = b0 + 32 * u + lane;
                    double e = 0.0;
                    if (idx < len) {
                        const int b = i + 1 + idx;
                        const double P1 = (i >= 1) ? tc[u] + pl[u] : 0.0;
                        double t = 2.0 * P1;
                        t = t - Pda;
                        t = t + vecB[b];
                        t = t - Prowa;
                        t = t - vecA[b];
                        e = t;
                        a.y[rs + idx] = t;
                    }
                    loc[u] = scan32_local(e, lane);
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {              // the carry chain
                    if (b0 + 32 * u < len) {
                        const int idx = b0 + 32 * u + lane;
                        const double out = carry + loc[u];
                        carry = __shfl_sync(0xffffffffu, out, 31);
                        if (idx < len) a.Rw[rs + idx] = out;
                    }
                }
            }
            if (lane == 0) a.RT[i] = carry;
        }
        if (gtid == 0) a.RT[n - 1] = 0.0;
        CG_MARK(6)
        grid_barrier(a.bar, nblocks, gen);   // phase 4 reads P/T of the first prefix and writes Rw/y/RT only; P/T are rewritten after this barrier
        CG_MARK(7)
        // ---- phase 5: k_colscan_local<true>
        for (long long idx = gtid; idx < (long long)nchunks * n; idx += gthreads)
            colscan_local_thread<true>(a.Rw, a.y, a.P, a.T, a.T2, n, (int)(idx / n), (int)(idx % n));
        CG_MARK(8)
        grid_barrier(a.bar, nblocks, gen);
        CG_MARK(9)
        // ---- phase 6: k_colscan_carry<true>
        for (long long j = gtid; j < n; j += gthreads) colscan_carry_thread<true>(a.T, a.T2, a.CT, n, nchunks, (int)j);
        CG_MARK(10)
        grid_barrier(a.bar, nblocks, gen);
        CG_MARK(11)
        // ---- phase 7 (per CTA): k_prs -> vecA; vecB[j] = G(j,j) = fixed G at (j-1, j)
        for (int j = tid; j < n; j += CGP_THREADS) {   // operands first (every load of the CTA in flight at once) ...
            vecA[j] = ldg_cg(a.RT + j) + ldg_cg(a.CT + j);
            vecB[j] = (j >= 1) ? fixed_P(a.P, a.T, n, j - 1, j) : 0.0;
        }
        __syncthreads();
        // ... then the blocked scan in place, from shared memory: every warp scans 32-blocks locally, one warp applies the
        // sequential carries (out_b = carry_b + local_b, carry_{b+1} = out_b[31]: k_prs's operands and order)
        for (int blk = (tid >> 5) * 32; blk < n; blk += CGP_THREADS) {
            const double e = (blk + lane < n) ? vecA[blk + lane] : 0.0;
            const double l = scan32_local(e, lane);
            if (blk + lane < n) vecA[blk + lane] = l;
        }
        __syncthreads();
        if (tid < 32) {
            double carry = 0.0;
            for (int blk = 0; blk < n; blk += 32) {
                const int last = min(blk + 31, n - 1);
                const double out = (blk + lane < n) ? carry + vecA[blk + lane] : 0.0;
                if (blk + lane < n) vecA[blk + lane] = out;
                // the block's last lane in k_prs is lane 31 of a zero-padded block: its value equals the last valid entry's
                carry = __shfl_sync(0xffffffffu, out, last - blk);
            }
        }
        __syncthreads();
        CG_MARK(12)
        // ---- phase 8: w = mask(A^T y), partial products p.w   (k_atx_combine<1>, fix folded in)
        for (long long vb0 = (long long)blockIdx.x * CGP_Q; vb0 < nblk; vb0 += (long long)gridDim.x * CGP_Q) {
            const long long vb = vb0 + g;
            const bool valid = vb < nblk;
            const int64_t base = (int64_t)vb * 1024 + 4 * t4;
            double prod[4] = {0.0, 0.0, 0.0, 0.0};
            if (valid && base < np) {
                int64_t i = (int64_t)(((2.0 * n - 1.0) - sqrt((2.0 * n - 1.0) * (2.0 * n - 1.0) - 8.0 * (double)base)) * 0.5);
                while (i > 0 && row_start(n, i) > base) --i;
                while (row_start(n, i + 1) <= base) ++i;
                int64_t j = base - row_start(n, i) + i + 1;
                // a thread's 4 consecutive entries share one 32-byte sector per array: the q = 0 loads go to L2, the rest hit L1
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int64_t kk = base + q;
                    if (kk < np) {
                        const double Gij = ldg_cg(a.T + (int64_t)((int)i / COL_CHUNK) * n + j) + ldg_cg(a.P + kk);
                        const double pk = ldg_cg(a.p + kk);
                        const bool act = a.active[kk] != 0;
                        const double u = vecA[j] - vecA[i];
                        const double wv = vecB[j] - Gij;
                        double pv = u - 2.0 * wv;
                        if (act) pv = 0.0;
                        prod[q] = pk * pv;
                        a.w[kk] = pv;
                        if (++j == n) { ++i; j = i + 1; }
                    }
                }
            }
            double s = ((prod[0] + prod[1]) + prod[2]) + prod[3];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) s = s + __shfl_xor_sync(0xffffffffu, s, off);
            if ((tid & 31) == 0) sh8[g][(tid >> 5) & 7] = s;
            __syncthreads();
            if (t4 == 0 && valid) {
                double t = sh8[g][0];
                for (int w = 1; w < 8; ++w) t = t + sh8[g][w];
                a.part1[vb] = t;
            }
            __syncthreads();
        }
        CG_MARK(13)
        grid_barrier(a.bar, nblocks, gen);
        CG_MARK(14)
        // ---- phase 9: EP_ALPHA
        dot = cgp_reduce(a.part1, nblk, lv, sh8, &bval);
        alpha = rho / dot;
        CG_MARK(15)
        // ---- phase 10: x += alpha p ; r -= alpha w ; partials r.r   (k_xr_update)
        for (long long vb0 = (long long)blockIdx.x * CGP_Q; vb0 < nblk; vb0 += (long long)gridDim.x * CGP_Q) {
            const long long vb = vb0 + g;
            const bool valid = vb < nblk;
            const int64_t base = (int64_t)vb * 1024 + 4 * t4;
            double e[4] = {0.0, 0.0, 0.0, 0.0};
            if (valid) {
                if (base + 3 < np) {   // 16-byte loads first (base is a multiple of 4: aligned), then the stores
                    const double2 x0 = *reinterpret_cast<const double2*>(a.x + base), x1 = *reinterpret_cast<const double2*>(a.x + base + 2);
                    const double2 p0 = *reinterpret_cast<const double2*>(a.p + base), p1 = *reinterpret_cast<const double2*>(a.p + base + 2);
                    const double2 r0 = *reinterpret_cast<const double2*>(a.r + base), r1 = *reinterpret_cast<const double2*>(a.r + base + 2);
                    const double2 w0 = *reinterpret_cast<const double2*>(a.w + base), w1 = *reinterpret_cast<const double2*>(a.w + base + 2);
                    double2 nx0, nx1, nr0, nr1;
                    nx0.x = x0.x + alpha * p0.x; nx0.y = x0.y + alpha * p0.y; nx1.x = x1.x + alpha * p1.x; nx1.y = x1.y + alpha * p1.y;
                    nr0.x = r0.x - alpha * w0.x; nr0.y = r0.y - alpha * w0.y; nr1.x = r1.x - alpha * w1.x; nr1.y = r1.y - alpha * w1.y;
                    *reinterpret_cast<double2*>(a.x + base) = nx0; *reinterpret_cast<double2*>(a.x + base + 2) = nx1;
                    *reinterpret_cast<double2*>(a.r + base) = nr0; *reinterpret_cast<double2*>(a.r + base + 2) = nr1;
                    e[0] = nr0.x * nr0.x; e[1] = nr0.y * nr0.y; e[2] = nr1.x * nr1.x; e[3] = nr1.y * nr1.y;
                } else {
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        if (base + q < np) {
                            const double xv = ldg_cg(a.x + base + q), pv = ldg_cg(a.p + base + q);
                            const double rv = ldg_cg(a.r + base + q), wv = ldg_cg(a.w + base + q);
                            a.x[base + q] = xv + alpha * pv;
                            const double nr = rv - alpha * wv;
                            a.r[base + q] = nr;
                            e[q] = nr * nr;
                        }
                }
            }
            double s = ((e[0] + e[1]) + e[2]) + e[3];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) s = s + __shfl_xor_sync(0xffffffffu, s, off);
            if ((tid & 31) == 0) sh8[g][(tid >> 5) & 7] = s;
            __syncthreads();
            if (t4 == 0 && valid) {
                double t = sh8[g][0];
                for (int w = 1; w < 8; ++w) t = t + sh8[g][w];
                a.part2[vb] = t;
            }
            __syncthreads();
        }
        CG_MARK(16)
        grid_barrier(a.bar, nblocks, gen);
        CG_MARK(17)
        // ---- phase 11: EP_RHO_STEP and the loop test (:796)
        const double val = cgp_reduce(a.part2, nblk, lv, sh8, &bval);
        rho_old = rho;
        iters_total += 1;
        rho = val;
        if ((val > e0sq) && (k < kmax)) { k += 1; if (k > 1) beta = val / rho_old; }
        else done = 1;
        CG_MARK(18)
        if (!done && a.max_iters > 0 && --left == 0) break;   // same decision in every CTA: resumable
    }
    if (gtid == 0) {
        a.sc->rho = rho; a.sc->rho_old = rho_old; a.sc->beta = beta; a.sc->alpha = alpha; a.sc->dot = dot;
        a.sc->k = k; a.sc->iters_total = iters_total; a.sc->done = done;
    }
    if (PROF && prof) {
#pragma unroll
        for (int q = 0; q < 20; ++q) a.prof[q] += tacc[PROF ? q : 0];
    }
#undef CG_MARK
}

// ============================================================================ literal-order path (parity ladder L0 on the device)
// opts.reserved[4] = 2.  The SAME arithmetic as CircularSplitWeights.java in the SAME order, so that the weights can be held
// bit for bit against the literal CPU restatement (oracle/nnet_oracle.cpp) - the check the production formulation above
// cannot give, because the active-set path is sensitive to summation order (SURVEY F5):
//   * calculateAb / calculateAtx as the reference's n-1 dependent diagonals (:603-633, :643-731): one CTA, one
//     __syncthreads per diagonal, each entry from the same three neighbours with the same operator order;
//   * rowsum (:571-591) one thread per row, strictly in index order;
//   * norm (:740-749) and the alpha dot (:815-817) as LEFT-TO-RIGHT sums, by the verified binade-collapsed exact
//     summation of fnn_exact_sum.cuh (bit-identical to `for (k) ss += x[k]*x[k]` for any signs);
//   * the whole loop of circularConjugateGrads (:769-831) in one single-CTA kernel.
// A validation mode: n <= 512 (one exact-summation block covers n(n-1)/2 <= 131072 addends), O(n) barriers per mat-vec.
namespace lit {
constexpr int THREADS = xsum::THREADS;
constexpr int MAX_N = 512;

__device__ double rowsum(int n, const double* d, int k) {   // :571-591
    double r = 0;
    int64_t index = 0;
    if (k > 0) {
        index = k - 1;
        for (int i = 0; i < k; i++) { r += d[index]; index += (n - i - 2); }
        index++;
    }
    for (int j = k + 1; j < n; j++) r += d[index++];
    return r;
}
// p = A^T d (:603-633); block-wide, p must not alias d
__device__ void atx(int n, const double* d, double* p) {
    const int tid = threadIdx.x;
    for (int i = tid; i < n - 1; i += THREADS) p[row_start(n, i)] = rowsum(n, d, i + 1);
    __syncthreads();
    for (int i = tid; i < n - 2; i += THREADS) {
        const int64_t index = row_start(n, i) + 1;
        p[index] = p[index - 1] + p[index + (n - i - 2)] - 2 * d[index + (n - i - 2)];
    }
    __syncthreads();
    for (int k = 3; k <= n - 1; k++) {
        for (int i = tid; i <= n - k - 1; i += THREADS) {
            const int64_t index = row_start(n, i) + (k - 1);
            p[index] = p[index - 1] + p[index + n - i - 2] - p[index + n - i - 3] - 2.0 * d[index + n - i - 2];
        }
        __syncthreads();
    }
}
// d = A b (:643-731); block-wide, d must not alias b
__device__ void ab(int n, const double* b, double* d) {
    const int tid = threadIdx.x;
    for (int i = tid; i <= n - 2; i += THREADS) {
        double d_ij = 0.0;
        int64_t index = i - 1;
        for (int k = 0; k <= i - 1; k++) { d_ij += b[index]; index += (n - k - 2); }
        index++;
        for (int k = i + 1; k <= n - 1; k++) d_ij += b[index++];
        d[row_start(n, i)] = d_ij;
    }
    __syncthreads();
    for (int i = tid; i <= n - 3; i += THREADS) {
        const int64_t index = row_start(n, i) + 1;
        d[index] = d[index - 1] + d[index + (n - i - 2)] - 2 * b[index - 1];
    }
    __syncthreads();
    for (int k = 3; k <= n - 1; k++) {
        for (int i = tid; i <= n - k - 1; i += THREADS) {
            const int64_t index = row_start(n, i) + (k - 1);
            d[index] = d[index - 1] + d[index + (n - i - 2)] - d[index + (n - i - 2) - 1] - 2.0 * b[index - 1];
        }
        __syncthreads();
    }
}
// sum_k f(k), k = 0..len-1, strictly left to right; result to every thread
template <typename F>
__device__ double seqsum(xsum::Smem* sm, int len, F f, double* res) {
    const int L = (len + xsum::THREADS - 1) / xsum::THREADS;
    auto load = [&](int, int t, int k) -> double { return f(t * L + k); };
    xsum::block_exact_seq_sum<1>(sm, len, load, [](int) { return true; }, res);
    __syncthreads();
    const double v = res[0];
    __syncthreads();
    return v;
}

__global__ void __launch_bounds__(THREADS, 1) k_matvec(int which, int n, const double* in, double* out) {
    if (which == 0) ab(n, in, out); else atx(n, in, out);
}

// circularConjugateGrads (:769-831), W == 1; one CTA runs the whole loop
__global__ void __launch_bounds__(THREADS, 1)
k_cg(int n, int np, double* r, double* w, double* p, double* y, const double* b, const unsigned char* active, double* x,
     Scalars* sc) {
    extern __shared__ unsigned char smem_raw[];
    xsum::Smem* sm = reinterpret_cast<xsum::Smem*>(smem_raw);
    __shared__ double res[1];
    const int tid = threadIdx.x;
    const long long kmax = sc->kmax;   // npairs, or the test budget of fnn_split_weights_budget
    ab(n, x, y);
    atx(n, y, r);
    for (int k = tid; k < np; k += THREADS) r[k] = active[k] ? 0.0 : b[k] - r[k];
    __syncthreads();
    double rho = seqsum(sm, np, [&](int k) { const double v = r[k]; return v * v; }, res);
    double rho_old = 0;
    const double e_0 = 1e-8 * sqrt(seqsum(sm, np, [&](int k) { const double v = b[k]; return v * v; }, res));
    long long k = 0;
    while ((rho > e_0 * e_0) && (k < kmax)) {
        k = k + 1;
        if (k == 1) { for (int i = tid; i < np; i += THREADS) p[i] = r[i]; }
        else {
            const double beta = rho / rho_old;
            for (int i = tid; i < np; i += THREADS) p[i] = r[i] + beta * p[i];
        }
        __syncthreads();
        ab(n, p, y);
        atx(n, y, w);
        for (int i = tid; i < np; i += THREADS) if (active[i]) w[i] = 0.0;
        __syncthreads();
        double alpha = seqsum(sm, np, [&](int i) { return p[i] * w[i]; }, res);
        alpha = rho / alpha;
        for (int i = tid; i < np; i += THREADS) { x[i] += alpha * p[i]; r[i] -= alpha * w[i]; }
        __syncthreads();
        rho_old = rho;
        rho = seqsum(sm, np, [&](int i) { const double v = r[i]; return v * v; }, res);
    }
    if (tid == 0) { sc->iters_total += k; sc->k = k; sc->rho = rho; sc->done = 1; }
}
}  // namespace lit

// ============================================================================ host driver
struct Csw {
    int n = 0;
    int64_t np = 0, nblk = 0;
    cudaStream_t st = nullptr;
    double *d = nullptr, *x = nullptr, *r = nullptr, *w = nullptr, *p = nullptr, *y = nullptr, *old_x = nullptr, *AtWd = nullptr;
    double *Rw = nullptr, *P = nullptr, *RT = nullptr, *CT = nullptr, *PRS = nullptr, *part1 = nullptr, *part2 = nullptr;
    double *T = nullptr, *T2 = nullptr;   // column-scan chunk totals / carries
    int nchunks = 0;
    unsigned char* active = nullptr;
    Scalars* sc = nullptr;
    Scalars* h_sc = nullptr;
    cudaGraphExec_t cg_graph = nullptr;
    int64_t cg_calls = 0, outer = 0, inner = 0, launches = 0, launches_per_graph = 0;
    // CG iteration cap of every circularConjugateGrads call (kmax of :795, uploaded to Scalars::kmax): npairs, or
    // min(npairs, max_cg_iters) under the budget of fnn_split_weights_budget; max_cg_calls > 0 stops the active-set method
    // right after that many CG calls.  0 = no budget (production).
    long long kmax = 0, max_cg_iters = 0, max_cg_calls = 0;
    bool budget_spent() const { return max_cg_calls > 0 && cg_calls >= max_cg_calls; }
    std::chrono::steady_clock::time_point t_start = std::chrono::steady_clock::now();
    double t_progress = 0.0;
    int persistent = 0;        // 1: k_cg_persistent (one cooperative launch per CG solve) instead of the graph path
    int persistent_grid = 0;
    unsigned long long* bar = nullptr;
    unsigned long long* prof = nullptr;   // FNN_CSW_PROF: per-phase ns of k_cg_persistent (CTA 0)
    int literal = 0;           // opts.reserved[4] == 2: the reference's own operation order (namespace lit), n <= 512
    // work arrays of the hand-written selection primitives (60 % collapse, argmins, split emission)
    SelState* sel = nullptr;
    SelState* h_sel = nullptr;          // pinned copy
    MinLoc* ml_part = nullptr;          // per-block partial min-locs
    int *tie_flag = nullptr, *tie_rank = nullptr;
    long long* blk_sum = nullptr;       // flag scan: per-1024-block counts -> exclusive offsets
    int sel_grid = 0;

    int* done_ptr() { return &sc->done; }

    int alloc() {
#define CSW_ALLOC(ptr, count) FNN_CUDA(cudaMalloc((void**)&(ptr), sizeof(*(ptr)) * (size_t)(count)))
        CSW_ALLOC(d, np); CSW_ALLOC(x, np); CSW_ALLOC(r, np); CSW_ALLOC(w, np); CSW_ALLOC(p, np); CSW_ALLOC(y, np);
        CSW_ALLOC(old_x, np); CSW_ALLOC(AtWd, np); CSW_ALLOC(Rw, np); CSW_ALLOC(P, np);
        CSW_ALLOC(RT, n); CSW_ALLOC(CT, n); CSW_ALLOC(PRS, n);
        nchunks = (n + COL_CHUNK - 1) / COL_CHUNK;
        CSW_ALLOC(T, (size_t)nchunks * n); CSW_ALLOC(T2, (size_t)nchunks * n);
        CSW_ALLOC(part1, nblk + 1); CSW_ALLOC(part2, nblk + 1);   // part2: level-2 scratch, or the r.r partials of k_cg_persistent
        CSW_ALLOC(bar, 2);
        if (getenv("FNN_CSW_PROF")) { CSW_ALLOC(prof, 24); FNN_CUDA(cudaMemset(prof, 0, 24 * sizeof(unsigned long long))); }
        CSW_ALLOC(active, np); CSW_ALLOC(sc, 1);
        sel_grid = (int)std::max<int64_t>(1, std::min<int64_t>((np + SEL_THREADS * 8 - 1) / (SEL_THREADS * 8), 148 * 4));
        CSW_ALLOC(tie_flag, np); CSW_ALLOC(tie_rank, np); CSW_ALLOC(blk_sum, nblk + 1);
        CSW_ALLOC(sel, 1); CSW_ALLOC(ml_part, sel_grid);
        FNN_CUDA(cudaMemset(sel, 0, sizeof(SelState)));
        FNN_CUDA(cudaMallocHost((void**)&h_sel, sizeof(SelState)));
        FNN_CUDA(cudaMallocHost((void**)&h_sc, sizeof(Scalars)));
        FNN_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        FNN_CUDA(cudaMemsetAsync(sc, 0, sizeof(Scalars), st));
        return FNN_OK;
    }
    void release() {
        if (cg_graph) cudaGraphExecDestroy(cg_graph);
        cudaFree(d); cudaFree(x); cudaFree(r); cudaFree(w); cudaFree(p); cudaFree(y); cudaFree(old_x); cudaFree(AtWd);
        cudaFree(T); cudaFree(T2); cudaFree(Rw); cudaFree(P); cudaFree(RT); cudaFree(CT); cudaFree(PRS); cudaFree(part1); cudaFree(part2);
        cudaFree(active); cudaFree(sc); cudaFree(bar); cudaFree(prof);
        cudaFree(tie_flag); cudaFree(tie_rank); cudaFree(blk_sum); cudaFree(sel); cudaFree(ml_part);
        if (h_sel) cudaFreeHost(h_sel);
        if (h_sc) cudaFreeHost(h_sc);
        if (st) cudaStreamDestroy(st);
    }
    int grid1d(int64_t len, int threads) const { return (int)std::min<int64_t>((len + threads - 1) / threads, 148 * 16); }
    dim3 grid_rows() const { return dim3((unsigned)std::max(1, std::min((n + 255) / 256, 64)), (unsigned)(n - 1)); }

    template <bool WITH_CT>
    void colscan(const double* in, const int* gate) {
        const dim3 g((unsigned)((n + 127) / 128), (unsigned)nchunks);
        k_colscan_local<WITH_CT><<<g, 128, 0, st>>>(Rw, in, P, T, T2, n, gate);
        k_colscan_carry<WITH_CT><<<(n + 127) / 128, 128, 0, st>>>(T, T2, CT, n, nchunks, gate);
        k_colscan_fix<<<grid_rows(), 256, 0, st>>>(P, T, n, gate);
    }
    // out = A in   (d = A b)
    void Ab(const double* in, double* out, const int* gate) {
        if (literal) { lit::k_matvec<<<1, lit::THREADS, 0, st>>>(0, n, in, out); launches += 1; return; }
        k_rowscan<<<std::min(n, 148 * 8), 256, 0, st>>>(in, Rw, nullptr, n, gate);
        colscan<false>(in, gate);
        k_ab_combine<<<grid_rows(), 256, 0, st>>>(P, out, n, gate);
        launches += 5;
    }
    // G/PRS for A^T in
    void Atx_prefix(const double* in, const int* gate) {
        k_rowscan<<<std::min(n, 148 * 8), 256, 0, st>>>(in, Rw, RT, n, gate);
        colscan<true>(in, gate);
        k_prs<<<1, 32, 0, st>>>(RT, CT, PRS, n, gate);
        launches += 5;
    }
    void Atx(const double* in, double* out, const int* gate) {
        if (literal) { lit::k_matvec<<<1, lit::THREADS, 0, st>>>(1, n, in, out); launches += 1; return; }
        Atx_prefix(in, gate);
        k_atx_combine<0><<<(unsigned)nblk, 256, 0, st>>>(P, PRS, out, n, np, nullptr, nullptr, nullptr, gate);
        launches += 1;
    }
    // reduce part1[0..nblk) with the fixed tree, finishing with epilogue ep
    void finish_tree(int ep, int gated) {
        const double* in = part1;
        double* out = part2;
        int64_t len = nblk;
        while (true) {
            const int64_t blocks = (len + 1023) / 1024;
            k_tree_level<<<(unsigned)blocks, 256, 0, st>>>(in, len, out, ep, sc, gated);
            launches += 1;
            if (blocks == 1) break;
            in = out; out = (out == part2) ? part1 : part2;   // part1 is free once consumed
            len = blocks;
        }
    }
    void cg_iteration() {   // one pass of the loop body (:797-829); all kernels no-op once sc->done
        k_pupdate<<<grid1d(np, 256), 256, 0, st>>>(p, r, np, sc);
        Ab(p, y, done_ptr());
        Atx_prefix(y, done_ptr());
        k_atx_combine<1><<<(unsigned)nblk, 256, 0, st>>>(P, PRS, w, n, np, active, p, part1, done_ptr());
        finish_tree(EP_ALPHA, 1);
        k_xr_update<<<(unsigned)nblk, 256, 0, st>>>(x, r, p, w, np, sc, part1);
        finish_tree(EP_RHO_STEP, 1);
        launches += 3;
    }
    // circularConjugateGrads (:769-831) with b = AtWd
    int conjugate_grads() {
        ++cg_calls;
        h_sc->k = 0;
        FNN_CUDA(cudaMemsetAsync(&sc->done, 0, sizeof(int), st));
        FNN_CUDA(cudaMemsetAsync(&sc->k, 0, sizeof(long long), st));
        if (literal) {
            lit::k_cg<<<1, lit::THREADS, sizeof(xsum::Smem), st>>>(n, (int)np, r, w, p, y, AtWd, active, x, sc);
            launches += 1;
            FNN_CUDA(cudaGetLastError());
            return FNN_OK;
        }
        Ab(x, y, nullptr);
        Atx(y, r, nullptr);
        k_residual_init<<<(unsigned)nblk, 256, 0, st>>>(r, AtWd, active, np, part1);
        finish_tree(EP_RHO_INIT, 0);
        launches += 1;
        if (persistent) {
            // bounded launches (the kernel is resumable: all loop state lives in Scalars and the barrier words)
            long long per_launch = 1 << 16;
            if (const char* e = getenv("FNN_CSW_ITERS_PER_LAUNCH")) per_launch = std::max<long long>(1, atoll(e));   // profiling sessions
            FNN_CUDA(cudaMemsetAsync(bar, 0, 2 * sizeof(unsigned long long), st));
            // FNN_CSW_ABORT_AFTER=<iterations>: measurement aid for sizes whose full solve does not fit a session - stop once
            // that many CG iterations have run, report the rate, fail the call (the weights are NOT a solution)
            static const long long abort_after = getenv("FNN_CSW_ABORT_AFTER") ? atoll(getenv("FNN_CSW_ABORT_AFTER")) : 0;
            static const double progress_every = getenv("FNN_CSW_PROGRESS") ? atof(getenv("FNN_CSW_PROGRESS")) : 0.0;   // seconds
            while (true) {
                FNN_CUDA(cudaMemcpyAsync(h_sc, sc, sizeof(Scalars), cudaMemcpyDeviceToHost, st));
                FNN_CUDA(cudaStreamSynchronize(st));
                if (h_sc->done) break;
                if (progress_every > 0.0) {
                    const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
                    if (secs - t_progress >= progress_every) {
                        t_progress = secs;
                        fprintf(stderr, "[fnn] split weights n=%d: %.0f s, %lld CG iterations, %lld CG solves, outer %lld, inner %lld\n", n, secs,
                                (long long)h_sc->iters_total, (long long)cg_calls, (long long)outer, (long long)inner);
                        fflush(stderr);
                    }
                }
                if (abort_after > 0 && h_sc->iters_total >= abort_after) {
                    const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
                    fprintf(stderr, "[fnn] split weights n=%d aborted on request after %lld CG iterations in %lld CG solves, %.2f s since the solve began "
                                    "(%.1f us per iteration all in)\n", n, (long long)h_sc->iters_total, (long long)cg_calls, secs,
                            1e6 * secs / (double)h_sc->iters_total);
                    fnn::set_error("split weights aborted after %lld CG iterations (FNN_CSW_ABORT_AFTER)", (long long)h_sc->iters_total);
                    return FNN_E_STATE;
                }
                CgArgs a{x, r, p, w, y, Rw, P, RT, CT, T, T2, part1, part2, active, sc, bar, n, nchunks, (long long)np, (long long)nblk, per_launch, prof};
                void* params[] = {&a};
                FNN_CUDA(cudaLaunchCooperativeKernel(prof ? (const void*)k_cg_persistent<true> : (const void*)k_cg_persistent<false>, dim3((unsigned)persistent_grid), dim3(CGP_THREADS), params,
                                                     sizeof(double) * 2 * (size_t)n, st));
                launches += 1;
            }
            return FNN_OK;
        }
        if (!cg_graph) {
            cudaGraph_t g;
            const int64_t before = launches;
            FNN_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
            for (int i = 0; i < 8; ++i) cg_iteration();
            FNN_CUDA(cudaStreamEndCapture(st, &g));
            launches_per_graph = launches - before;
            launches = before;
            FNN_CUDA(cudaGraphInstantiate(&cg_graph, g, 0));
            cudaGraphDestroy(g);
        }
        while (true) {
            FNN_CUDA(cudaMemcpyAsync(h_sc, sc, sizeof(Scalars), cudaMemcpyDeviceToHost, st));
            FNN_CUDA(cudaStreamSynchronize(st));
            if (h_sc->done) break;
            for (int rep = 0; rep < 4; ++rep) { FNN_CUDA(cudaGraphLaunch(cg_graph, st)); launches += launches_per_graph; }
        }
        return FNN_OK;
    }
};

template <typename InOp>
static int minloc_reduce(Csw& c, InOp op, MinLoc* out_host) {
    k_minloc<InOp><<<c.sel_grid, SEL_THREADS, 0, c.st>>>(op, c.np, c.ml_part, c.sel);
    c.launches += 1;
    FNN_CUDA(cudaMemcpyAsync(c.h_sel, c.sel, sizeof(SelState), cudaMemcpyDeviceToHost, c.st));
    FNN_CUDA(cudaStreamSynchronize(c.st));
    out_host->v = c.h_sel->ml_v; out_host->i = c.h_sel->ml_i;
    return FNN_OK;
}

// worstIndices(x, 0.6) + contraction (:282-330, :420-431); returns whether anything was contracted.  Entirely on the device
// (count, exact radix select of the cutoff, marking, tie ranking by a flag scan); the host reads one counter at the end.
static int contract_worst(Csw& c, bool* contracted) {
    FNN_CUDA(cudaMemsetAsync(&c.sel->num_neg, 0, sizeof(long long), c.st));
    k_sel_count_neg<<<c.sel_grid, SEL_THREADS, 0, c.st>>>(c.x, c.np, c.sel);
    for (int pass = 0; pass < 8; ++pass) k_sel_radix_pass<<<c.sel_grid, SEL_THREADS, 0, c.st>>>(c.x, c.np, c.sel, pass);
    k_sel_mark<<<c.grid1d(c.np, 256), 256, 0, c.st>>>(c.x, c.active, c.np, c.sel, c.tie_flag);
    // more ties at the cutoff than slots left (rare): rank the ties in index order, the earliest fill the slots
    k_flag_local<<<(unsigned)c.nblk, 1024, 0, c.st>>>(c.tie_flag, c.np, c.tie_rank, c.blk_sum, c.sel);
    k_flag_blockscan<<<1, 1024, 0, c.st>>>(c.blk_sum, c.nblk, c.sel, c.sel);
    k_sel_mark_ties<<<c.grid1d(c.np, 256), 256, 0, c.st>>>(c.x, c.active, c.np, c.sel, c.tie_flag, c.tie_rank, c.blk_sum);
    c.launches += 13;
    FNN_CUDA(cudaMemcpyAsync(c.h_sel, c.sel, sizeof(SelState), cudaMemcpyDeviceToHost, c.st));
    FNN_CUDA(cudaStreamSynchronize(c.st));
    *contracted = c.h_sel->num_neg > 0;
    return FNN_OK;
}

// runActiveConjugate (:359-557)
static int active_conjugate(Csw& c) {
    const int n = c.n;
    k_unconstrained<<<c.grid_rows(), 256, 0, c.st>>>(c.d, c.x, n);
    MinLoc ml;
    {   // all_positive test (:369-374): any x < 0 ?
        if (minloc_reduce(c, RatioIn{c.x, c.x}, &ml)) return FNN_E_CUDA;   // only the index matters here
        if (ml.i < 0) return FNN_OK;
    }
    k_fill<<<c.grid1d(c.np, 256), 256, 0, c.st>>>(c.old_x, c.np, 1.0);
    FNN_CUDA(cudaMemsetAsync(c.active, 0, c.np, c.st));
    c.Atx(c.d, c.AtWd, nullptr);   // y = W*d = d
    // e_0 depends only on b = AtWd: compute once (the literal path recomputes it, left to right, in lit::k_cg)
    if (!c.literal) {
        k_square_partials<<<(unsigned)c.nblk, 256, 0, c.st>>>(c.AtWd, c.np, c.part1);
        c.finish_tree(EP_E0, 0);
    }
    c.kmax = c.max_cg_iters > 0 ? std::min<long long>(c.np, c.max_cg_iters) : (long long)c.np;
    FNN_CUDA(cudaMemcpyAsync(&c.sc->kmax, &c.kmax, sizeof(long long), cudaMemcpyHostToDevice, c.st));
    bool first_pass = true;
    while (true) {
        ++c.outer;
        while (true) {
            ++c.inner;
            if (!first_pass) {
                if (c.conjugate_grads()) return FNN_E_CUDA;
                if (c.budget_spent()) return FNN_OK;
            }
            first_pass = false;
            bool contracted = false;
            if (contract_worst(c, &contracted)) return FNN_E_CUDA;
            if (contracted) {
                if (c.conjugate_grads()) return FNN_E_CUDA;
                if (c.budget_spent()) return FNN_OK;
            }
            if (minloc_reduce(c, RatioIn{c.x, c.old_x}, &ml)) return FNN_E_CUDA;
            if (ml.i < 0) break;
            k_oldx_step<<<c.grid1d(c.np, 256), 256, 0, c.st>>>(c.old_x, c.x, c.active, c.np, ml.v);
            k_set_one<<<1, 32, 0, c.st>>>(c.x, c.active, ml.i, 0.0, 1, 1);
            c.launches += 2;
        }
        c.Ab(c.x, c.y, nullptr);
        c.Atx(c.y, c.r, nullptr);
        k_gradient<<<c.grid1d(c.np, 256), 256, 0, c.st>>>(c.r, c.AtWd, c.np);
        if (minloc_reduce(c, GradIn{c.r, c.active}, &ml)) return FNN_E_CUDA;
        if (ml.i < 0 || ml.v > -0.0000001) return FNN_OK;
        k_set_one<<<1, 32, 0, c.st>>>(c.x, c.active, ml.i, 0.0, 0, 0);
    }
}

}  // namespace

extern "C" int fnn_csw_matvec(const fnn_opts* o, int32_t which, const double* v, int64_t n, double* out) {
    if (!v || !out || n < 4 || n > 20000) { fnn::set_error("fnn_csw_matvec: bad arguments"); return FNN_E_ARG; }
    int cnt = 0;
    if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt <= 0) { cudaGetLastError(); fnn::set_error("no CUDA device available (libfastnn has no CPU fallback)"); return FNN_E_NODEVICE; }
    FNN_CUDA(cudaSetDevice(o ? o->device : 0));
    Csw c;
    c.n = (int)n; c.np = n * (n - 1) / 2; c.nblk = (c.np + 1023) / 1024;
    c.literal = (o && o->reserved[4] == 2) ? 1 : 0;
    if (c.literal && n > lit::MAX_N) { fnn::set_error("fnn_csw_matvec: the literal-order validation mode covers n <= %d", lit::MAX_N); return FNN_E_ARG; }
    int rc = c.alloc();
    if (!rc) {
        cudaMemcpyAsync(c.x, v, sizeof(double) * c.np, cudaMemcpyHostToDevice, c.st);
        if (which == 0) c.Ab(c.x, c.y, nullptr);
        else if (which == 1) c.Atx(c.x, c.y, nullptr);
        else k_unconstrained<<<c.grid_rows(), 256, 0, c.st>>>(c.x, c.y, c.n);
        cudaMemcpyAsync(out, c.y, sizeof(double) * c.np, cudaMemcpyDeviceToHost, c.st);
        if (cudaStreamSynchronize(c.st) != cudaSuccess || cudaGetLastError() != cudaSuccess) {
            fnn::set_error("fnn_csw_matvec: %s", cudaGetErrorString(cudaGetLastError()));
            rc = FNN_E_CUDA;
        }
    }
    c.release();
    return rc;
}

// allocation and solver configuration for n taxa, once per workspace
static int csw_prepare(Csw& c, const fnn_opts* o, int64_t n) {
    c.n = (int)n; c.np = n * (n - 1) / 2; c.nblk = (c.np + 1023) / 1024;
    c.literal = (o && o->reserved[4] == 2) ? 1 : 0;
    if (c.literal && n > lit::MAX_N) { fnn::set_error("split weights: the literal-order validation mode covers n <= %d", lit::MAX_N); return FNN_E_ARG; }
    int rc = c.alloc();
    if (rc) return rc;
    if (c.literal) FNN_CUDA(cudaFuncSetAttribute(lit::k_cg, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(xsum::Smem)));
    if (!c.literal && !(o && o->reserved[4] == 1) && n <= CGP_MAX_N) {   // reserved[4] = 1 keeps the launch-per-phase graph path (A/B)
        int dev = 0, coop = 0, sms = 0, per_sm = 0;
        FNN_CUDA(cudaGetDevice(&dev));
        FNN_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
        FNN_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        FNN_CUDA(cudaFuncSetAttribute(k_cg_persistent<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double) * 2 * (size_t)n)));
        FNN_CUDA(cudaFuncSetAttribute(k_cg_persistent<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double) * 2 * (size_t)n)));
        FNN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_cg_persistent<true>, CGP_THREADS, sizeof(double) * 2 * (size_t)n));
        per_sm = std::min(per_sm, 1);
        if (coop && per_sm >= 1) {
            c.persistent = 1;
            int64_t want = (c.np + 2047) / 2048;   // >= 4 entries per thread and phase; fewer CTAs = cheaper barriers
            if (const char* e = getenv("FNN_CSW_GRID")) want = atoll(e);
            c.persistent_grid = (int)std::max<int64_t>(1, std::min<int64_t>((int64_t)sms * per_sm, want));
        }
    }
    return FNN_OK;
}

// a prepared workspace back in the state csw_prepare leaves it in, for the next solve of the same size
static int csw_reset(Csw& c) {
    FNN_CUDA(cudaMemsetAsync(c.sc, 0, sizeof(Scalars), c.st));
    FNN_CUDA(cudaMemsetAsync(c.sel, 0, sizeof(SelState), c.st));
    memset(c.h_sc, 0, sizeof(Scalars));
    c.cg_calls = c.outer = c.inner = c.launches = 0;
    return FNN_OK;
}

// upload, permute to circular-position order, solve; leaves x on the device
static int csw_solve(Csw& c, const fnn_opts* o, const int32_t* ordering, const double* d_upper, bool d_upper_on_device) {
    const int64_t n = c.n;
    int* d_ord = reinterpret_cast<int*>(c.tie_rank);   // scratch: free until the first 60 % collapse
    FNN_CUDA(cudaMemcpyAsync(d_ord, ordering, sizeof(int) * (n + 1), cudaMemcpyHostToDevice, c.st));
    FNN_CUDA(cudaMemcpyAsync(c.r, d_upper, sizeof(double) * c.np, d_upper_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice,
                             c.st));   // r as staging
    k_setup_d<<<c.grid_rows(), 256, 0, c.st>>>(c.r, d_ord, c.d, c.n);
    const bool unconstrained = o && o->reserved[3] == 1;
    if (unconstrained) {
        k_unconstrained<<<c.grid_rows(), 256, 0, c.st>>>(c.d, c.x, c.n);
        return FNN_OK;
    }
    return active_conjugate(c);
}

// shared driver of the B2 entry points; leaves x on the device
static int solve_split_weights(Csw& c, const fnn_opts* o, const int32_t* ordering, const double* d_upper, int64_t n) {
    int rc = csw_prepare(c, o, n);
    if (rc) return rc;
    return csw_solve(c, o, ordering, d_upper, false);
}

static int check_b2_args(const fnn_opts* o, const int32_t* ordering, const double* d_upper, int64_t n) {
    if (!ordering || !d_upper || n < 4 || n > 20000) { fnn::set_error("split weights: bad arguments (4 <= n <= 20000)"); return FNN_E_ARG; }
    int cnt = 0;
    if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt <= 0) { cudaGetLastError(); fnn::set_error("no CUDA device available (libfastnn has no CPU fallback)"); return FNN_E_NODEVICE; }
    FNN_CUDA(cudaSetDevice(o ? o->device : 0));
    return FNN_OK;
}

static int fetch_stats(Csw& c, int64_t* stats_out) {
    FNN_CUDA(cudaMemcpyAsync(c.h_sc, c.sc, sizeof(Scalars), cudaMemcpyDeviceToHost, c.st));
    FNN_CUDA(cudaStreamSynchronize(c.st));
    FNN_CUDA(cudaGetLastError());
    if (c.prof && c.h_sc->iters_total > 0) {
        unsigned long long h[24];
        FNN_CUDA(cudaMemcpy(h, c.prof, sizeof(h), cudaMemcpyDeviceToHost));
        static const char* nm[19] = {"ph1 pupdate+rowscan", "bar1", "ph2 colscan_local", "bar2", "ph3 carry", "bar3", "ph4 combine+rowscan", "bar4",
                                     "ph5 colscan_local+CT", "bar5", "ph6 carry+CT", "bar6", "ph7 prs+diag", "ph8 atx combine+dot", "bar7",
                                     "ph9 reduce alpha", "ph10 xr update", "bar8", "ph11 reduce rho"};
        double tot = 0;
        for (int q = 0; q < 19; ++q) tot += (double)h[q];
        fprintf(stderr, "[fnn] k_cg_persistent n=%d grid=%d: %.2f us per iteration over %lld iterations (CTA 0):\n", c.n, c.persistent_grid,
                tot / 1e3 / (double)c.h_sc->iters_total, (long long)c.h_sc->iters_total);
        for (int q = 0; q < 19; ++q) fprintf(stderr, "[fnn]   %-24s %7.2f us\n", nm[q], (double)h[q] / 1e3 / (double)c.h_sc->iters_total);
    }
    if (stats_out) { stats_out[0] = c.h_sc->iters_total; stats_out[1] = c.cg_calls; stats_out[2] = c.outer; stats_out[3] = c.inner; stats_out[4] = c.launches; }
    return FNN_OK;
}

extern "C" int fnn_split_weights(const fnn_opts* o, const int32_t* ordering, const double* d_upper, int64_t n, double* x_out,
                                 int64_t* stats_out) {
    int rc = check_b2_args(o, ordering, d_upper, n);
    if (rc) return rc;
    if (!x_out) { fnn::set_error("fnn_split_weights: null output"); return FNN_E_ARG; }
    Csw c;
    rc = solve_split_weights(c, o, ordering, d_upper, n);
    if (!rc && cudaMemcpyAsync(x_out, c.x, sizeof(double) * c.np, cudaMemcpyDeviceToHost, c.st) != cudaSuccess) {
        fnn::set_error("fnn_split_weights: %s", cudaGetErrorString(cudaGetLastError()));
        rc = FNN_E_CUDA;
    }
    if (!rc) rc = fetch_stats(c, stats_out);
    c.release();
    return rc;
}

extern "C" int fnn_split_weights_budget(const fnn_opts* o, const int32_t* ordering, const double* d_upper, int64_t n,
                                        int64_t max_cg_iters, int64_t max_cg_calls, double* x_out, uint8_t* active_out,
                                        int64_t* stats_out) {
    int rc = check_b2_args(o, ordering, d_upper, n);
    if (rc) return rc;
    if (!x_out || !active_out || max_cg_iters < 0 || max_cg_calls < 0) {
        fnn::set_error("fnn_split_weights_budget: null output or negative budget");
        return FNN_E_ARG;
    }
    Csw c;
    c.max_cg_iters = max_cg_iters;
    c.max_cg_calls = max_cg_calls;
    rc = solve_split_weights(c, o, ordering, d_upper, n);
    if (!rc) {
        // the mask is set up when the active-set loop is entered (outer > 0); before that every split is free
        if (c.outer == 0) memset(active_out, 0, (size_t)c.np);
        if (cudaMemcpyAsync(x_out, c.x, sizeof(double) * c.np, cudaMemcpyDeviceToHost, c.st) != cudaSuccess ||
            (c.outer > 0 && cudaMemcpyAsync(active_out, c.active, (size_t)c.np, cudaMemcpyDeviceToHost, c.st) != cudaSuccess)) {
            fnn::set_error("fnn_split_weights_budget: %s", cudaGetErrorString(cudaGetLastError()));
            rc = FNN_E_CUDA;
        }
    }
    if (!rc) rc = fetch_stats(c, stats_out);
    c.release();
    return rc;
}

// (:94-108 / FastNN.java:455-466) keep x > cutoff, in (i,j) row-major-upper order - compacted on the device (flag scan of the
// selection primitives above) so that only the ~3.7 n surviving splits cross PCIe instead of n(n-1)/2 weights (SURVEY §8f N2)
__global__ void k_flag_above(const double* __restrict__ x, int* __restrict__ flag, int64_t len, double cutoff) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x) flag[i] = x[i] > cutoff;
}
// compaction in index order: flagged entry i goes to slot block_excl[i / 1024] + local_rank[i]
__global__ void k_compact(const double* __restrict__ x, const int* __restrict__ flag, const int* __restrict__ local_rank,
                          const long long* __restrict__ block_excl, int64_t len, int* __restrict__ idx_out, double* __restrict__ w_out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x)
        if (flag[i]) {
            const long long k = block_excl[i >> 10] + local_rank[i];
            idx_out[k] = (int)i;
            w_out[k] = x[i];
        }
}

// FastNN.java:455-466 on the device: flag the splits whose weight exceeds `cutoff` and count them (one host read)
static int count_kept(Csw& c, double cutoff, long long* kept) {
    k_flag_above<<<c.grid1d(c.np, 256), 256, 0, c.st>>>(c.x, c.tie_flag, c.np, cutoff);
    k_flag_local<<<(unsigned)c.nblk, 1024, 0, c.st>>>(c.tie_flag, c.np, c.tie_rank, c.blk_sum, nullptr);
    k_flag_blockscan<<<1, 1024, 0, c.st>>>(c.blk_sum, c.nblk, c.sel, nullptr);
    FNN_CUDA(cudaMemcpyAsync(c.h_sel, c.sel, sizeof(SelState), cudaMemcpyDeviceToHost, c.st));
    FNN_CUDA(cudaStreamSynchronize(c.st));
    *kept = c.h_sel->flag_total;
    return FNN_OK;
}

// the solver's scratch vectors are free now: the first kept ints of w get the flagged packed indices in (i, j) order,
// p their weights
static int* compact_kept(Csw& c) {
    int* d_idx = reinterpret_cast<int*>(c.w);
    k_compact<<<c.grid1d(c.np, 256), 256, 0, c.st>>>(c.x, c.tie_flag, c.tie_rank, c.blk_sum, c.np, d_idx, c.p);
    return d_idx;
}

// the compacted splits to the host as (i, j, weight)
static int copy_kept(Csw& c, int64_t n, long long kept, int32_t* split_i, int32_t* split_j, double* weight) {
    if (kept <= 0) return FNN_OK;
    std::vector<int> idx_h((size_t)kept);
    FNN_CUDA(cudaMemcpyAsync(idx_h.data(), c.w, sizeof(int) * (size_t)kept, cudaMemcpyDeviceToHost, c.st));
    FNN_CUDA(cudaMemcpyAsync(weight, c.p, sizeof(double) * (size_t)kept, cudaMemcpyDeviceToHost, c.st));
    FNN_CUDA(cudaStreamSynchronize(c.st));
    int64_t i = 0;
    for (long long k = 0; k < kept; ++k) {   // packed index -> (i, j); indices are increasing, so i only moves forward
        while (row_start(n, i + 1) <= idx_h[k]) ++i;
        split_i[k] = (int32_t)i;
        split_j[k] = (int32_t)(idx_h[k] - row_start(n, i) + i + 1);
    }
    return FNN_OK;
}

// keep x > cutoff, compacted in (i, j) order, and copy them out
static int emit_kept_splits(Csw& c, int64_t n, double cutoff, int32_t* split_i, int32_t* split_j, double* weight, int64_t max_out,
                            int64_t* n_out) {
    long long kept = 0;
    int rc = count_kept(c, cutoff, &kept);
    if (rc) return rc;
    *n_out = kept;
    if (kept > max_out) { fnn::set_error("weighted splits: %lld splits kept, room for %lld", kept, (long long)max_out); return FNN_E_ARG; }
    if (kept > 0) compact_kept(c);
    return copy_kept(c, n, kept, split_i, split_j, weight);
}

extern "C" int fnn_weighted_splits(const fnn_opts* o, const int32_t* ordering, const double* d_upper, int64_t n, double cutoff,
                                   int32_t* split_i, int32_t* split_j, double* weight, int64_t max_out, int64_t* n_out,
                                   int64_t* stats_out) {
    int rc = check_b2_args(o, ordering, d_upper, n);
    if (rc) return rc;
    if (!split_i || !split_j || !weight || !n_out || max_out < 0) { fnn::set_error("fnn_weighted_splits: null output"); return FNN_E_ARG; }
    Csw c;
    rc = solve_split_weights(c, o, ordering, d_upper, n);
    if (!rc) {
        rc = emit_kept_splits(c, n, cutoff, split_i, split_j, weight, max_out, n_out);
    }
    if (!rc) rc = fetch_stats(c, stats_out);
    c.release();
    return rc;
}

// packed upper triangle (DistancesAndNames order) of an n x ld device matrix
__global__ void k_pack_upper(const double* __restrict__ D, int64_t ld, int n, double* __restrict__ out) {
    const int i = blockIdx.y;
    if (i > n - 2) return;
    const int64_t rs = (int64_t)i * (2 * n - i - 1) / 2;
    for (int j = i + 1 + blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) out[rs + (j - i - 1)] = D[(int64_t)i * ld + j];
}

// FastNN.main's ordering stage and split stage chained with the distances kept on the device (fnn_network, fnn_bootstrap):
// the packed upper triangle is taken from the device matrix before the ordering consumes it, so the split stage uploads
// nothing but the ordering.  The workspace serves every run of the same n.
struct NetChain {
    fnn_opts o;
    int64_t n = 0;
    Csw c;
    double* d_upper = nullptr;
    bool used = false;
};

int fnn_chain_create_(const fnn_opts* o, int64_t n, NetChain** out) {
    NetChain* w = new NetChain();
    if (o) w->o = *o;
    else fnn_default_opts(&w->o);
    w->n = n;
    int rc = csw_prepare(w->c, &w->o, n);
    if (!rc && cudaMalloc((void**)&w->d_upper, sizeof(double) * (size_t)w->c.np) != cudaSuccess) {
        fnn::set_error("split weights: cudaMalloc of the packed triangle failed: %s", cudaGetErrorString(cudaGetLastError()));
        rc = FNN_E_CUDA;
    }
    if (rc) { fnn_chain_destroy_(w); return rc; }
    *out = w;
    return FNN_OK;
}

void fnn_chain_destroy_(NetChain* w) {
    if (!w) return;
    w->c.release();
    if (w->d_upper) cudaFree(w->d_upper);
    delete w;
}

int fnn_chain_run_(NetChain* w, fnn_ctx* ctx, double cutoff, int32_t* ordering_out, int64_t* kept, ChainTimes* tm) {
    const int64_t n = w->n;
    Csw& c = w->c;
    double* dD; int64_t ld;
    fnn_ctx_matrix_ptr(ctx, &dD, &ld);
    cudaStream_t cs = fnn_ctx_stream_(ctx);
    DevEvent p0, p1, s0, s1;
    if (tm) {
        FNN_CUDA(p0.create()); FNN_CUDA(p1.create()); FNN_CUDA(s0.create()); FNN_CUDA(s1.create());
        FNN_CUDA(cudaEventRecord(p0, cs));
    }
    k_pack_upper<<<dim3((unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, 64)), (unsigned)(n - 1)), 256, 0, cs>>>(dD, ld, (int)n, w->d_upper);
    FNN_CUDA(cudaGetLastError());
    if (tm) FNN_CUDA(cudaEventRecord(p1, cs));
    FNN_CUDA(cudaStreamSynchronize(cs));
    int rc = fnn_ctx_order(ctx, ordering_out);
    if (rc) return rc;
    if (w->used) { rc = csw_reset(c); if (rc) return rc; }
    w->used = true;
    if (tm) FNN_CUDA(cudaEventRecord(s0, c.st));
    rc = csw_solve(c, &w->o, ordering_out, w->d_upper, true);
    if (rc) return rc;
    long long k = 0;
    rc = count_kept(c, cutoff, &k);
    if (rc) return rc;
    *kept = k;
    if (k > 0) compact_kept(c);
    FNN_CUDA(cudaGetLastError());
    if (tm) {
        FNN_CUDA(cudaEventRecord(s1, c.st));
        FNN_CUDA(cudaMemcpyAsync(c.h_sc, c.sc, sizeof(Scalars), cudaMemcpyDeviceToHost, c.st));
        FNN_CUDA(cudaStreamSynchronize(c.st));
        fnn_stats st;
        fnn_ctx_stats(ctx, &st);
        float a = 0, b = 0;
        cudaEventElapsedTime(&a, p0, p1);
        cudaEventElapsedTime(&b, s0, s1);
        tm->order_ms = st.order_ms;
        tm->csw_ms = (double)a + (double)b;
        tm->cg_iters = c.h_sc->iters_total;
    }
    return FNN_OK;
}

const int* fnn_chain_kept_idx_(NetChain* w) { return reinterpret_cast<const int*>(w->c.w); }
cudaStream_t fnn_chain_stream_(NetChain* w) { return w->c.st; }
int fnn_chain_copy_kept_(NetChain* w, int64_t kept, int32_t* split_i, int32_t* split_j, double* weight) {
    return copy_kept(w->c, w->n, kept, split_i, split_j, weight);
}

// The whole network in one call (SURVEY §8b "optional fnn_network").
extern "C" int fnn_network(const fnn_opts* o, const double* D_rowmajor, int64_t n, double cutoff, int32_t* ordering_out,
                           int32_t* split_i, int32_t* split_j, double* weight, int64_t max_out, int64_t* n_out) {
    if (!D_rowmajor || !ordering_out || !split_i || !split_j || !weight || !n_out || n < 4 || n > 20000) {
        fnn::set_error("fnn_network: bad arguments (4 <= n <= 20000)");
        return FNN_E_ARG;
    }
    fnn_ctx* ctx = nullptr;
    int rc = fnn_ctx_create(o, n, &ctx);
    if (rc) return rc;
    NetChain* w = nullptr;
    rc = fnn_ctx_load_host(ctx, D_rowmajor);
    if (!rc) rc = fnn_chain_create_(o, n, &w);
    int64_t kept = 0;
    if (!rc) rc = fnn_chain_run_(w, ctx, cutoff, ordering_out, &kept, nullptr);
    if (!rc) {
        *n_out = kept;
        if (kept > max_out) {
            fnn::set_error("weighted splits: %lld splits kept, room for %lld", (long long)kept, (long long)max_out);
            rc = FNN_E_ARG;
        } else {
            rc = fnn_chain_copy_kept_(w, kept, split_i, split_j, weight);
        }
    }
    fnn_chain_destroy_(w);
    fnn_ctx_destroy(ctx);
    return rc;
}
