// fnn_modes.cuh — the Relaxed and Random selection strategies (SURVEY §8 a14, a16) on the device.
// Included by fnn_order.cu inside its anonymous namespace (needs DevState).
//
//   Random  (NeighborNetRandom.java:31-48, :130-178): k_random_walk generates the reference's
//           java.util.Random walk in parallel by speculation, k_random_eval evaluates the sampled Q
//           values on all SMs and reduces on (Q, draw index) = "first strict minimum in draw order".
//   Relaxed (NeighborNetLocal.java:88-264): k_relaxed_select - one lane runs the control flow as a
//           resumable state machine (fnn_relaxed_sm.h), the block does the row scans (findRowMin,
//           :88-126) and the -additive look-ahead (:280-466) it asks for.
#pragma once
#include "fnn_relaxed_sm.h"
#include "fnn_record.h"

namespace modes {

constexpr int THREADS = 1024;
constexpr int MAX_TIES = 4096;

// ---- java.util.Random on the device -------------------------------------------------------
__device__ __forceinline__ int jr_next(unsigned long long& s, int bits) {
    s = (s * 0x5DEECE66DULL + 0xBULL) & ((1ULL << 48) - 1);
    return (int)((long long)s >> (48 - bits));
}
__device__ inline int jr_next_int(unsigned long long& s, int bound) {
    int r = jr_next(s, 31);
    const int m = bound - 1;
    if ((bound & m) == 0) return (int)(((long long)bound * (long long)r) >> 31);
    for (int u = r;; u = jr_next(s, 31)) {
        r = u % bound;
        if ((int)((unsigned)u - (unsigned)r + (unsigned)m) >= 0) break;   // Java int wrap-around
    }
    return r;
}

// cluster distance with the reference's role order: p first, q second (e.g. NeighborNetRandom.java:161-168)
__device__ __forceinline__ double dpq_roles(const double* __restrict__ D, int64_t ld, int sp, int sq, int P2) {
    const int spn = sp < P2 ? (sp ^ 1) : -1, sqn = sq < P2 ? (sq ^ 1) : -1;
    const double* rp = D + (int64_t)sp * ld;
    if (spn < 0 && sqn < 0) return rp[sq];
    if (spn >= 0 && sqn < 0) return (rp[sq] + D[(int64_t)spn * ld + sq]) * 0.5;
    if (spn < 0) return (rp[sq] + rp[sqn]) * 0.5;
    const double* rpn = D + (int64_t)spn * ld;
    return (((rp[sq] + rp[sqn]) + rpn[sq]) + rpn[sqn]) * 0.25;
}

// ceil(log10(total)) as Java computes it (Math.log10 is exact on powers of ten): smallest k with 10^k >= total
__device__ __forceinline__ int ceil_log10(int total) {
    int k = 0;
    long long p = 1;
    while (p < total) { p *= 10; ++k; }
    return k;
}

// ---------------------------------------------------------------- Random findNodes
// The walk of NeighborNetRandom.java:140-158 is a chain: draw k uses bound m-1 or m-2 depending on whether the
// node reached by draw k-1 is paired, nextInt(bound) may reject (consuming more LCG steps), and j is remapped when
// it hits i or i.nbr.  k_random_walk still generates it in PARALLEL, by speculation:
//   * raw 31-bit values for a window of draws by LCG jump-ahead (one LCG step per draw if nothing rejects);
//   * both candidates (mod m-1, mod m-2) per draw; "is the reached node paired" is a 2-state automaton whose
//     per-draw transition functions are composed with a block-wide scan;
//   * rejections and remaps are rare (~bound/2^31 and ~2/m per draw): the first one in the window is found with
//     a min-reduce, everything before it is committed, that single draw is replayed exactly by one lane, and the
//     window restarts behind it.
// The committed (i, j) pairs go to global memory; k_random_eval evaluates Q for them on all SMs and reduces on
// (Q, draw index) = "first strict minimum in draw order" (:172-176).
constexpr unsigned long long JR_A = 0x5DEECE66DULL, JR_C = 0xBULL, JR_MASK = (1ULL << 48) - 1;
constexpr int WALK_G = 8;                       // draws per thread per window
constexpr int WALK_W = THREADS * WALK_G;        // window

// first-try result of java.util.Random.nextInt(bound) for the raw 31-bit value u
__device__ __forceinline__ int jr_cand(int u, int bound) {
    return (bound & (bound - 1)) == 0 ? (int)(((long long)bound * (long long)u) >> 31) : u % bound;
}

struct WalkState { long long count; long long total; int cur; int pad; };

// state after k LCG steps: s -> A^k s + C (A^k - 1)/(A - 1)   (mod 2^48), by binary decomposition of k
__device__ __forceinline__ unsigned long long jr_jump(unsigned long long s, unsigned k, const unsigned long long* Ap,
                                                      const unsigned long long* Cp) {
    for (int b = 0; k; ++b, k >>= 1)
        if (k & 1) s = (Ap[b] * s + Cp[b]) & JR_MASK;
    return s;
}

__device__ __forceinline__ long long random_search_amount(int mode, int mult, int m) {   // findSearchAmount (:31-48)
    long long amount;
    if (mode == 4) amount = ceil_log10(m);
    else if (mode == 2) amount = m;
    else amount = (long long)ceil_log10(m) * m;
    return (long long)mult * amount;
}

__global__ void __launch_bounds__(THREADS, 1)
k_random_walk(const int* __restrict__ pos, const int* __restrict__ p2s, DevState* st, int* __restrict__ nbrpos,
              int2* __restrict__ pairs, WalkState* ws, long long* __restrict__ record) {
    if (st->done || st->mode < 2 || st->m <= st->fallback) return;
    __shared__ unsigned long long Ap[24], Cp[24];
    __shared__ unsigned char wfun[THREADS / 32];
    __shared__ int wlast[THREADS / 32];
    __shared__ int wexc[THREADS / 32];
    __shared__ unsigned long long s_base;
    __shared__ int s_cur, s_exc;
    __shared__ long long s_count;
    __shared__ long long s_rejected, s_remapped;   // strategy record (only when one is kept)
    const int m = st->m, P2 = st->P2, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long total = random_search_amount(st->mode, st->mult, m);
    if (tid == 0) tl_stamp(st, TL_SCAN0);
    // neighbour position per position (-1: singleton), shared by this kernel's parallel lookups
    for (int i = tid; i < m; i += THREADS) {
        const int s = p2s[i];
        nbrpos[i] = s < P2 ? pos[s ^ 1] : -1;
    }
    if (tid == 0) {
        unsigned long long a = JR_A, c = JR_C;
        for (int b = 0; b < 24; ++b) { Ap[b] = a; Cp[b] = c; c = (c * (a + 1)) & JR_MASK; a = (a * a) & JR_MASK; }
        unsigned long long rng = st->rng;
        s_cur = jr_next_int(rng, m);   // int i = myRandom.nextInt(num_active) (:134)
        s_base = rng;
        s_count = 0;
        s_rejected = s_remapped = 0;
    }
    __syncthreads();   // also publishes nbrpos (block-local producer/consumer through global memory)
    __threadfence_block();
    while (true) {
        const long long count = s_count;
        if (count >= total) break;
        const unsigned long long base = s_base;
        const int cur0 = s_cur;
        const int wlen = (int)min((long long)WALK_W, total - count);
        const int d0 = tid * WALK_G;
        // ---- raw values + both candidates of my draws
        int ra[WALK_G], ca[WALK_G], cb[WALK_G];
        unsigned long long sst = (d0 < wlen) ? jr_jump(base, (unsigned)d0, Ap, Cp) : 0ull;
        unsigned f0 = 0, f1 = 1;   // composed transition so far: state in -> state out
#pragma unroll
        for (int g = 0; g < WALK_G; ++g) {
            if (d0 + g < wlen) {
                sst = (sst * JR_A + JR_C) & JR_MASK;
                const int u = (int)(sst >> 17);
                ra[g] = u;
                ca[g] = jr_cand(u, m - 1);   // candidate when the current node is a singleton
                cb[g] = jr_cand(u, m - 2);   // candidate when it is paired
                const unsigned pa = nbrpos[ca[g]] >= 0, pb = nbrpos[cb[g]] >= 0;
                // compose: new f(x) = (old f(x) ? pb : pa)
                f0 = f0 ? pb : pa;
                f1 = f1 ? pb : pa;
            }
        }
        // ---- block-wide composition scan of the 2-state transition functions (exclusive)
        unsigned c0 = f0, c1 = f1;   // inclusive composition within the warp
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const unsigned p0 = __shfl_up_sync(0xffffffffu, c0, off), p1 = __shfl_up_sync(0xffffffffu, c1, off);
            if (lane >= off) { const unsigned n0 = p0 ? c1 : c0, n1 = p1 ? c1 : c0; c0 = n0; c1 = n1; }   // (prev then mine)
        }
        if (lane == 31) wfun[warp] = (unsigned char)(c0 | (c1 << 1));
        __syncthreads();
        // incoming state of this thread = composition of everything before it applied to the start state
        unsigned st_in = nbrpos[cur0] >= 0;
        for (int w = 0; w < warp; ++w) st_in = (wfun[w] >> st_in) & 1u;
        {
            const unsigned e0 = __shfl_up_sync(0xffffffffu, c0, 1), e1 = __shfl_up_sync(0xffffffffu, c1, 1);
            if (lane > 0) st_in = st_in ? e1 : e0;
        }
        // ---- replay my draws: chosen candidate, exceptions
        int jj[WALK_G];
        int myexc = 0x7fffffff, mylast = -1;
        unsigned sx = st_in;
#pragma unroll
        for (int g = 0; g < WALK_G; ++g) {
            if (d0 + g < wlen) {
                const int bound = sx ? (m - 2) : (m - 1);
                const int j = sx ? cb[g] : ca[g];
                jj[g] = j;
                if ((bound & (bound - 1)) != 0 && (int)((unsigned)ra[g] - (unsigned)j + (unsigned)(bound - 1)) < 0)
                    myexc = min(myexc, d0 + g);   // nextInt would reject and draw again
                sx = nbrpos[j] >= 0;
                mylast = j;
            }
        }
        if (lane == 31 || d0 + WALK_G >= wlen) { /* last j of the warp is published below */ }
        // previous draw's j (= my first i): from the previous thread, or cur0
        int prevj = __shfl_up_sync(0xffffffffu, mylast, 1);
        if (lane == 31) wlast[warp] = mylast;
        __syncthreads();
        if (lane == 0) prevj = (warp == 0) ? cur0 : wlast[warp - 1];
        int ii = prevj;
#pragma unroll
        for (int g = 0; g < WALK_G; ++g) {
            if (d0 + g < wlen) {
                const int inb = nbrpos[ii];
                if (jj[g] == ii || (inb >= 0 && jj[g] == inb)) myexc = min(myexc, d0 + g);   // remap cases (:144-157)
                ii = jj[g];
            }
        }
        for (int off = 16; off > 0; off >>= 1) myexc = min(myexc, __shfl_xor_sync(0xffffffffu, myexc, off));
        if (lane == 0) wexc[warp] = myexc;
        __syncthreads();
        if (tid == 0) {
            int e = wexc[0];
            for (int w = 1; w < THREADS / 32; ++w) e = min(e, wexc[w]);
            s_exc = e;
        }
        __syncthreads();
        const int exc = min(s_exc, wlen);   // draws [0, exc) are exactly the reference's
        // ---- commit
        ii = prevj;
#pragma unroll
        for (int g = 0; g < WALK_G; ++g) {
            if (d0 + g < exc) pairs[count + d0 + g] = make_int2(ii, jj[g]);
            if (d0 + g < wlen) ii = jj[g];
        }
        // new walk position = j of draw exc-1
        if (exc > 0 && d0 <= exc - 1 && exc - 1 < d0 + WALK_G) s_cur = jj[exc - 1 - d0];
        __syncthreads();
        if (tid == 0) {
            unsigned long long rng = jr_jump(base, (unsigned)exc, Ap, Cp);
            long long done_n = exc;
            if (exc < wlen) {   // replay the exceptional draw exactly
                const int i = s_cur;
                const int inb = nbrpos[i];
                const unsigned long long one_step = (rng * JR_A + JR_C) & JR_MASK;
                int j, j0;
                if (inb >= 0) {
                    j = j0 = jr_next_int(rng, m - 2);
                    if (i == j && m - 1 == inb) j = m - 2;
                    else if (i == j && m - 1 != inb) j = m - 1;
                    else if (inb == j && m - 2 == i) j = m - 1;
                    else if (inb == j && m - 2 != i) j = m - 2;
                } else {
                    j = j0 = jr_next_int(rng, m - 1);
                    if (i == j) j = m - 1;
                }
                if (record) {   // the exception was a rejection (nextInt took more than one LCG step), a remap, or both
                    s_rejected += rng != one_step;
                    s_remapped += j != j0;   // every remap target lies outside nextInt's range, so a remap always changes j
                }
                pairs[count + exc] = make_int2(i, j);
                s_cur = j;
                done_n += 1;
            }
            s_base = rng;
            s_count = count + done_n;
        }
        __syncthreads();
    }
    if (tid == 0) {
        st->rng = s_base;
        ws->count = s_count;
        ws->total = total;
        if (record) {   // k_random_eval adds the digest (column 3)
            long long* row = record + rec::COLS * (int64_t)st->iter;
            row[0] = s_count; row[1] = s_rejected; row[2] = s_remapped;
        }
    }
}

// Q for every committed pair, min-loc on (Q, draw index); the last block reduces the partials
__global__ void __launch_bounds__(256)
k_random_eval(const double* __restrict__ D, int64_t ld, const double* __restrict__ Sx, const int* __restrict__ p2s,
              DevState* st, const int2* __restrict__ pairs, const WalkState* ws, Partial* partials, unsigned int* ticket,
              long long* __restrict__ record) {
    if (st->done || st->mode < 2 || st->m <= st->fallback) return;
    __shared__ double wq[8];
    __shared__ unsigned long long wk[8];
    __shared__ bool amLast;
    const int P2 = st->P2, tid = threadIdx.x;
    const double cm2 = (double)st->c - 2.0;
    const long long total = ws->count;
    double bq = INFINITY;
    unsigned long long bk = ~0ull;
    unsigned long long abytes = 0;   // SURVEY 8(d) K9: 8*(1|2|4) + 16 bytes per sample
    unsigned long long digest = 0;   // strategy record: this thread's share of the draws' digest (fnn_record.h)
    for (long long k = (long long)blockIdx.x * blockDim.x + tid; k < total; k += (long long)gridDim.x * blockDim.x) {
        const int2 pr = pairs[k];
        if (record) digest += rec::draw_term(k, pr.x, pr.y);
        const int sp = p2s[pr.x], sq = p2s[pr.y];
        abytes += 8ull * (unsigned)((1 + (sp < P2)) * (1 + (sq < P2))) + 16ull;
        const double q = (cm2 * dpq_roles(D, ld, sp, sq, P2) - Sx[sp]) - Sx[sq];
        if (bk == ~0ull || q < bq || (q == bq && (unsigned long long)k < bk)) { bq = q; bk = (unsigned long long)k; }
    }
    auto take = [&](double oq, unsigned long long ok) {
        if (ok != ~0ull && (bk == ~0ull || oq < bq || (oq == bq && ok < bk))) { bq = oq; bk = ok; }
    };
    for (int off = 16; off > 0; off >>= 1) {
        const double oq = __shfl_down_sync(0xffffffffu, bq, off);
        const unsigned long long ok = __shfl_down_sync(0xffffffffu, bk, off);
        take(oq, ok);
    }
    for (int off = 16; off > 0; off >>= 1) abytes += __shfl_down_sync(0xffffffffu, abytes, off);
    if ((tid & 31) == 0) { wq[tid >> 5] = bq; wk[tid >> 5] = bk; if (abytes) atomicAdd(&st->strat_bytes, abytes); }
    if (record) {   // a sum mod 2^64: the order in which the warps add their shares does not matter
        for (int off = 16; off > 0; off >>= 1) digest += __shfl_down_sync(0xffffffffu, digest, off);
        if ((tid & 31) == 0 && digest)
            atomicAdd(reinterpret_cast<unsigned long long*>(record + rec::COLS * (int64_t)st->iter + 3), digest);
    }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < 8; ++w) take(wq[w], wk[w]);
        partials[blockIdx.x] = Partial{bq, bk};
        __threadfence();
        amLast = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (amLast && tid == 0) {
        __threadfence();
        bq = INFINITY; bk = ~0ull;
        for (int b = 0; b < (int)gridDim.x; ++b) take(__ldcg(&partials[b].q), __ldcg(&partials[b].key));
        const int2 pr = pairs[bk];
        st->cx_pos = pr.x;   // Cx = p, Cy = q (:173-176)
        st->cy_pos = pr.y;
        st->strat_units += (unsigned long long)total;
        *ticket = 0;
        tl_stamp(st, TL_SCAN1);
    }
}

// ---------------------------------------------------------------- Relaxed findRowMin (block-wide device function)
// Scans row `ip` over ALL active positions (NeighborNetLocal.java:100-126), writes the positions of every exact tie of
// the minimum, in position order, to out[0..count) (global memory) and returns count (or -1 if more than `room`).
__device__ int block_rowmin(const double* __restrict__ D, int64_t ld, const double* __restrict__ Sx, const int* __restrict__ pos,
                            const int* __restrict__ p2s, int m, int P2, double cm2, int ip, int* out, int room) {
    __shared__ double wmin[THREADS / 32];
    __shared__ int spos[MAX_TIES];
    __shared__ double gmin;
    __shared__ int cnt;
    const int tid = threadIdx.x;
    const int sp = p2s[ip];
    const int spn = sp < P2 ? (sp ^ 1) : -1;
    const double Sp = Sx[sp];
    const double* rp = D + (int64_t)sp * ld;
    const double* rpn = spn >= 0 ? D + (int64_t)spn * ld : rp;
    // Q(p, q) with p first (calculateDpq, NeighborNetLocal.java:266-278), every operand of a group of RU candidates loaded
    // before the first use: a row scan is a handful of rounds of independent loads, not one round per candidate
    constexpr int RU = 4;
    auto q_of = [&](int sq, double a, double b, double c2, double d2, double Sq) -> double {
        const bool qp = sq < P2;
        double dpq;
        if (spn < 0 && !qp) dpq = a;
        else if (spn >= 0 && !qp) dpq = (a + c2) * 0.5;          // (D[p][q] + D[p.nbr][q]) / 2
        else if (spn < 0) dpq = (a + b) * 0.5;                    // (D[p][q] + D[p][q.nbr]) / 2
        else dpq = (((a + b) + c2) + d2) * 0.25;                  // D[p][q] + D[p][q.nbr] + D[p.nbr][q] + D[p.nbr][q.nbr]
        return (cm2 * dpq - Sp) - Sq;
    };
    // the minimum and the SET of its ties do not depend on the visiting order, so the block walks physical slots
    // (coalesced rows) and orders the ties by position afterwards.  One pass: every thread keeps its minimum, the first
    // slot that reached it and how many of its candidates tie with it.
    double mn = INFINITY;
    int first_sq = -1, neq = 0;
    for (int s0 = tid; s0 < m; s0 += RU * THREADS) {
        double a[RU], b[RU], c2[RU], d2[RU], Sq[RU];
        bool use[RU];
#pragma unroll
        for (int u = 0; u < RU; ++u) {
            const int sq = s0 + u * THREADS;
            use[u] = sq < m && sq != sp && sq != spn;           // every active q except p and p.nbr (:100-105)
            a[u] = b[u] = c2[u] = d2[u] = Sq[u] = 0.0;
            if (use[u]) {
                const int sqn = sq < P2 ? (sq ^ 1) : sq;
                Sq[u] = Sx[sq]; a[u] = rp[sq]; b[u] = rp[sqn]; c2[u] = rpn[sq]; d2[u] = rpn[sqn];
            }
        }
#pragma unroll
        for (int u = 0; u < RU; ++u) {
            if (!use[u]) continue;
            const int sq = s0 + u * THREADS;
            const double q = q_of(sq, a[u], b[u], c2[u], d2[u], Sq[u]);
            if (q < mn) { mn = q; first_sq = sq; neq = 1; }
            else if (q == mn) { if (first_sq < 0) first_sq = sq; ++neq; }
        }
    }
    const double mine = mn;
    for (int off = 16; off > 0; off >>= 1) mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, off));
    if ((tid & 31) == 0) wmin[tid >> 5] = mn;
    if (tid == 0) cnt = 0;
    __syncthreads();
    if (tid == 0) {
        double g = wmin[0];
        for (int w = 1; w < THREADS / 32; ++w) g = fmin(g, wmin[w]);
        gmin = g;
    }
    __syncthreads();
    const double g = gmin;
    if (first_sq >= 0 && mine == g) {   // all exact ties (:118-124), gathered then ordered by position
        if (neq == 1) {
            const int k = atomicAdd(&cnt, 1);
            if (k < MAX_TIES) spos[k] = pos[first_sq];
        } else {                         // several ties inside this thread's candidates: walk them again
            for (int sq = tid; sq < m; sq += THREADS) {
                if (sq == sp || sq == spn) continue;
                const int sqn = sq < P2 ? (sq ^ 1) : sq;
                const double q = q_of(sq, rp[sq], rp[sqn], rpn[sq], rpn[sqn], Sx[sq]);
                if (q == g) {
                    const int k = atomicAdd(&cnt, 1);
                    if (k < MAX_TIES) spos[k] = pos[sq];
                }
            }
        }
    }
    __syncthreads();
    const int total = cnt;
    const int nt = min(total, MAX_TIES);
    if (tid == 0) {
        for (int a = 1; a < nt; ++a) {   // insertion sort: the list has one or two entries in practice
            const int v = spos[a];
            int b = a - 1;
            while (b >= 0 && spos[b] > v) { spos[b + 1] = spos[b]; --b; }
            spos[b + 1] = v;
        }
    }
    __syncthreads();
    if (total > MAX_TIES || total > room) return -1;
    for (int k = tid; k < nt; k += THREADS) out[k] = spos[k];
    __syncthreads();
    return nt;
}

// ---------------------------------------------------------------- Relaxed -additive look-ahead (block-wide device function)
// findAgglomeratedQ (NeighborNetLocal.java:280-386) with agg3wayLocal (:388-414) / agg4wayLocal (:416-466):
// simulate joining (Cx, Cy) and compare the Q of the merged cluster against testNode with the Q before the join
// (:241-247).  Cx, Cy are taken as selected (no id swap, as in the reference call at :245).  Returns (in thread 0)
// whether |originalQ - newQ| < 1e-7.
__device__ bool block_lookahead(const double* __restrict__ D, int64_t ld, const double* __restrict__ Sx, const int* __restrict__ p2s,
                                int m, int c, int P2, int cx_pos, int cy_pos, int test_pos, xsum::Smem* xs) {
    __shared__ double rx[4], crs[1];
    __shared__ int sh[2];
    const int tid = threadIdx.x;
    const int Cx = p2s[cx_pos], Cy = p2s[cy_pos], T = p2s[test_pos];
    const int Cxn = Cx < P2 ? (Cx ^ 1) : -1, Cyn = Cy < P2 ? (Cy ^ 1) : -1;
    const int L = (m + xsum::THREADS - 1) / xsum::THREADS;
    auto d = [&](int a, int b) -> double { return D[(int64_t)a * ld + b]; };
    const int zs[4] = {Cx, Cxn, Cy, Cyn};
    if (Cxn >= 0 || Cyn >= 0) {
        auto load = [&](int r, int t, int k) -> double {
            const int s = p2s[t * L + k];
            const double v = d(zs[r], s);
            const bool full = (s >= P2) || s == Cx || s == Cxn || s == Cy || s == Cyn;
            return full ? v : v * 0.5;
        };
        xsum::block_exact_seq_sum<4>(xs, m, load, [&](int r) { return zs[r] >= 0; }, rx);
    } else {
        if (tid < 4) rx[tid] = 0.0;
        __syncthreads();
    }
    if (tid == 0) {   // the 4-candidate pick (:311-335)
        int x = Cx, y = Cy;
        const double f = (double)(c + (Cxn >= 0) + (Cyn >= 0)) - 2.0;
        double best = (f * d(Cx, Cy) - rx[0]) - rx[2];
        if (Cxn >= 0) { const double q = (f * d(Cxn, Cy) - rx[1]) - rx[2]; if (q < best) { x = Cxn; y = Cy; best = q; } }
        if (Cyn >= 0) { const double q = (f * d(Cx, Cyn) - rx[0]) - rx[3]; if (q < best) { x = Cx; y = Cyn; best = q; } }
        if (Cxn >= 0 && Cyn >= 0) { const double q = (f * d(Cxn, Cyn) - rx[1]) - rx[3]; if (q < best) { x = Cxn; y = Cyn; best = q; } }
        sh[0] = x; sh[1] = y;
    }
    __syncthreads();
    const int x = sh[0], y = sh[1];
    const int xn = x < P2 ? (x ^ 1) : -1, yn = y < P2 ? (y ^ 1) : -1;
    int kind, X = -1, Y = -1, Z = -1, W = -1;
    if (xn < 0 && yn < 0) kind = 2;
    else if (xn < 0) { kind = 3; X = x; Y = y; Z = yn; }
    else if (yn < 0 || m == 4) { kind = 3; X = y; Y = x; Z = xn; }
    else { kind = 4; X = xn; Y = x; Z = y; W = yn; }   // (x2, x, y, y2)
    const double TT = 2.0 / 3.0;
    auto term = [&](int i) -> double {   // the per-position contribution to clusterRowSum
        const int p = p2s[i];
        const bool pair = p < P2;
        if (pair && (p & 1)) return 0.0;                       // not a representative
        const int pn = pair ? p + 1 : -1;
        if (kind == 2) {
            if (p == x || p == y) return 0.0;
            if (!pair) return (d(p, x) + d(p, y)) * 0.5;
            return (((d(p, x) + d(p, y)) + d(pn, x)) + d(pn, y)) * 0.25;
        } else if (kind == 3) {
            if (p == X || p == Y || p == Z || pn == Y || pn == Z) return 0.0;
            const double Dup = TT * d(X, p) + d(Y, p) / 3.0, Dvp = TT * d(Z, p) + d(Y, p) / 3.0;
            if (!pair) return (Dup + Dvp) * 0.5;
            const double Duq = TT * d(X, pn) + d(Y, pn) / 3.0, Dvq = TT * d(Z, pn) + d(Y, pn) / 3.0;
            return (((Dup + Dvp) + Duq) + Dvq) * 0.25;
        } else {
            if (p == X || p == Y || p == Z || p == W || pn == X || pn == Y || pn == Z || pn == W) return 0.0;
            const double Dup = TT * d(X, p) + d(Y, p) / 3.0, Dvp = TT * d(Z, p) + d(Y, p) / 3.0;
            const double Dup2 = TT * Dup + Dvp / 3.0, Dvp2 = TT * d(W, p) + Dvp / 3.0;
            if (!pair) return (Dup2 + Dvp2) * 0.5;
            const double Duq = TT * d(X, pn) + d(Y, pn) / 3.0, Dvq = TT * d(Z, pn) + d(Y, pn) / 3.0;
            const double Duq2 = TT * Duq + Dvq / 3.0, Dvq2 = TT * d(W, pn) + Dvq / 3.0;
            return (((Dup2 + Dvp2) + Duq2) + Dvq2) * 0.25;
        }
    };
    auto load1 = [&](int, int t, int k) -> double { return term(t * L + k); };
    xsum::block_exact_seq_sum<1>(xs, m, load1, [](int) { return true; }, crs);
    bool accept = false;
    if (tid == 0) {
        const double dCxT = dpq_roles(D, ld, Cx, T, P2), dCyT = dpq_roles(D, ld, Cy, T, P2);
        const double subtracted = (Sx[T] - dCxT) - dCyT;                                  // :337
        double cd;
        if (kind == 2) {
            const int Tn = T < P2 ? (T ^ 1) : -1;
            // calculateClusterDistLocal(x, testNode) (:349, :468-476); a singleton testNode makes the JAR throw there -
            // the oracle's documented substitute is the 2-term form against (x, y)
            cd = Tn >= 0 ? (d(x, T) + d(x, Tn)) * 0.5 : (d(T, x) + d(T, y)) * 0.5;
        } else cd = term(test_pos);
        const double A = ((double)c - 1.0) - 2.0;
        const double newQ = (A * cd - crs[0]) - (subtracted + cd);                        // :361 / :412 / :464
        const double origQ = (((double)c - 2.0) * dCxT - Sx[Cx]) - Sx[T];                 // :241-243
        accept = fabs(origQ - newQ) < .0000001;                                            // :247
    }
    return accept;
}

// ---------------------------------------------------------------- Relaxed findNodes: one kernel per iteration
// One lane advances the control state machine of fnn_relaxed_sm.h (the code the CPU tests hold against the literal
// oracle); whenever it asks for a row scan or a look-ahead, the whole block does it and resumes the machine.  No host
// round trip: Relaxed is as device-resident and graph-replayable as the other modes.
struct DevNodeView {
    const int* id; const int* pos; const int* p2s; int m_, P2;
    __device__ int m() const { return m_; }
    __device__ int id_at(int p) const { return id[p2s[p]]; }
    __device__ int nbr_pos(int p) const { const int s = p2s[p]; return s < P2 ? pos[s ^ 1] : -1; }
};

__global__ void __launch_bounds__(THREADS, 1)
k_relaxed_select(const double* __restrict__ D, int64_t ld, const double* __restrict__ Sx, const int* __restrict__ id,
                 const int* __restrict__ pos, const int* __restrict__ p2s, DevState* st, relaxed::Machine* Mg, int ntax,
                 long long* __restrict__ record) {
    if (st->done || st->mode != 1 || st->m <= st->fallback) return;
    extern __shared__ unsigned char smem_raw[];
    xsum::Smem* xs = reinterpret_cast<xsum::Smem*>(smem_raw);
    __shared__ relaxed::Machine M;
    __shared__ int req, look_accept;
    __shared__ long long s_rec[rec::COLS];   // strategy record (only when one is kept): scans, ties, look-aheads, digest
    const int m = st->m, c = st->c, P2 = st->P2, tid = threadIdx.x;
    const double cm2 = (double)c - 2.0;
    const DevNodeView nv{id, pos, p2s, m, P2};
    if (tid == 0) {
        tl_stamp(st, TL_SCAN0);   // timeline: the strategy kernel takes the scan's slots while m > fallback
        M = *Mg;
        relaxed::begin_call(M, ntax);
        look_accept = 0;
        for (int k = 0; k < rec::COLS; ++k) s_rec[k] = 0;
    }
    __syncthreads();
    while (true) {
        if (tid == 0) req = (int)relaxed::step(M, nv, look_accept);
        __syncthreads();
        const int r = req;
        if (r == relaxed::REQ_DONE || r == relaxed::REQ_ERROR) break;
        if (r == relaxed::REQ_SCAN) {
            const int cnt = block_rowmin(D, ld, Sx, pos, p2s, m, P2, cm2, M.req_pos, M.tiepool + M.tie_used, relaxed::tie_room(M));
            if (tid == 0) {
                // SURVEY 8(d) K7: a row scan reads the row (two rows if p is paired) and Sx
                st->strat_bytes += 8ull * (unsigned long long)m * (unsigned)(1 + (p2s[M.req_pos] < P2)) + 8ull * (unsigned long long)m;
                st->strat_units += 1;
                if (record) {   // block_rowmin has sorted the ties and written them (visible after its last barrier)
                    const int s = (int)s_rec[0];
                    unsigned long long dg = rec::scan_term(s, M.req_pos, -1, 0);
                    for (int r = 0; r < cnt; ++r) dg += rec::scan_term(s, M.req_pos, r, M.tiepool[M.tie_used + r]);
                    s_rec[0] += 1;
                    if (cnt > 0) s_rec[1] += cnt;
                    s_rec[3] = (long long)((unsigned long long)s_rec[3] + dg);
                }
                if (cnt < 0) M.error = 3;
                else relaxed::commit_scan(M, cnt);
            }
        } else {
            const bool acc = block_lookahead(D, ld, Sx, p2s, m, c, P2, M.cx_pos, M.cy_pos, M.look_test_pos, xs);
            if (tid == 0) { look_accept = acc ? 1 : 0; s_rec[2] += 1; }
        }
        __threadfence_block();
        __syncthreads();
        if (M.error) break;
    }
    if (tid == 0) {
        st->cx_pos = M.cx_pos;
        st->cy_pos = M.cy_pos;
        if (M.error || M.cx_pos < 0 || M.cy_pos < 0) { st->error = 10 + M.error; st->done = 1; st->skip = 1; }
        *Mg = M;
        if (record)
            for (int k = 0; k < rec::COLS; ++k) record[rec::COLS * (int64_t)st->iter + k] = s_rec[k];
        tl_stamp(st, TL_SCAN1);
    }
}

}  // namespace modes
