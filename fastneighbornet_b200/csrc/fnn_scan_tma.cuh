// fnn_scan_tma.cuh — K2, the selection scan, as a TMA-fed shared-memory pipeline (sm_100a).
//
// One persistent CTA per SM: a producer warp issues 2-D tiled TMA loads (cp.async.bulk.tensor,
// SASS UTMALDG) of 8-row x 256-column boxes of the distance matrix into a 6-stage ring
// (6 x 32 KB), completion signalled through mbarriers; eight consumer warps evaluate
// Q = (c-2)*Dpq - Sx[p] - Sx[q] on the staged rows and keep a per-thread (Q, i, j) min-loc.
// Memory-level parallelism comes from the ring (up to 192 KB in flight per SM), not from
// registers or occupancy.  From 4 096 active nodes up, k_prune (fnn_order.cu) first marks the row segments (one row, or one
// pair row, x 256 columns) whose lower bound on Q exceeds a Q already reached by a real pair; the scan then fetches only the
// surviving segments (1 x 256 boxes, or the two 8 x 256 boxes when a whole chunk survives) and reads the others' rows as
// Sx = -inf.  Included by fnn_order.cu (needs DevState, Partial, better()).
#pragma once
#include <cuda.h>
#include "fnn_tile_iter.h"

namespace tma {

constexpr int NGROUPS = 2;                  // consumer groups; group g owns rows [g*RPG, (g+1)*RPG) of every chunk
constexpr int GROUP = 256;                  // threads per group: one 16-byte column pair each
constexpr int CONSUMERS = GROUP * NGROUPS;  // 16 consumer warps
constexpr int THREADS = CONSUMERS + 32;     // + 1 producer warp
constexpr int BOX_W = 256;                  // TMA box: 256 columns (2 KB) ...
constexpr int BOX_R = 8;                    // ... x 8 rows
constexpr int RPG = BOX_R / NGROUPS;        // rows per consumer group per chunk (even)
static_assert(TILE_COLS == 2 * BOX_W && TILE_ROWS == 4 * BOX_R, "tile = 2 boxes wide, 4 chunks high");
constexpr int STAGES = 6;
constexpr int STAGE_BYTES = 2 * BOX_R * BOX_W * 8;   // 32 KB
constexpr size_t SMEM_BYTES = (size_t)STAGES * STAGE_BYTES + 1024;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int x, int y, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(dst)),
        "l"(map), "r"(x), "r"(y), "r"(smem_u32(bar))
        : "memory");
}

struct __align__(16) RowData { double S; long long pos; };   // one LDS.128 per row

#define FNN_CONSIDER(QV, RP, CP, ROWP)                                                                   \
    if ((QV) <= bq) {                                                                                    \
        const unsigned long long key_ = (ROWP) ? (((unsigned long long)(RP) << 32) | (unsigned)(CP))     \
                                               : (((unsigned long long)(CP) << 32) | (unsigned)(RP));    \
        if (better((QV), key_, bq, bk)) { bq = (QV); bk = key_; }                                        \
    }

__device__ __forceinline__ double2 lds2(const double* p) { return *reinterpret_cast<const double2*>(p); }

// Interior evaluators: "filter, then verify".  The hot loop evaluates a role-free approximation
// q~ = fma(c-2, Dpq~, -Sx[row]) - Sx[col] (fixed summation order, FMA allowed) and only tests
// q~ <= best + delta, where delta bounds |q~ - q| for the exactly rounded, role-ordered q of the
// reference (delta = 16*2^-53 * (3c+2) * max|D| + (c+2) * 2^-1074, DESIGN.md §4.1).  Groups that pass are re-walked
// with the exact arithmetic and the (Q, i, j) key, so the result is bit-identical to evaluating
// every entry exactly; on non-degenerate data the verify branch is taken a handful of times.
__device__ __forceinline__ void exact1(double e, const RowData r, double cm2, double cS, int cP, double& bq,
                                       unsigned long long& bk) {
    const int rp = (int)r.pos;
    const bool rowP = rp > cP;
    const double q = (cm2 * e - (rowP ? r.S : cS)) - (rowP ? cS : r.S);
    FNN_CONSIDER(q, rp, cP, rowP)
}
__device__ __forceinline__ void exact_pp(double2 e0, double2 e1, const RowData r, double cm2, double cS, int cP, double& bq,
                                         unsigned long long& bk) {
    const int rp = (int)r.pos;
    const bool rowP = rp > cP;
    const double dpq = (((e0.x + (rowP ? e0.y : e1.x)) + (rowP ? e1.x : e0.y)) + e1.y) * 0.25;
    const double q = (cm2 * dpq - (rowP ? r.S : cS)) - (rowP ? cS : r.S);
    FNN_CONSIDER(q, rp, cP, rowP)
}

// OR of (q[k] <= bound) as one chained DSETP per value (nvcc would otherwise rewrite the OR of
// compares into a tree of emulated fp64 minima, ~6 instructions each).
__device__ __forceinline__ bool any_le8(const double* q, double b) {
    int r;
    asm("{\n.reg .pred p;\n"
        "setp.le.f64 p, %1, %9;\n setp.le.or.f64 p, %2, %9, p;\n setp.le.or.f64 p, %3, %9, p;\n setp.le.or.f64 p, %4, %9, p;\n"
        "setp.le.or.f64 p, %5, %9, p;\n setp.le.or.f64 p, %6, %9, p;\n setp.le.or.f64 p, %7, %9, p;\n setp.le.or.f64 p, %8, %9, p;\n"
        "selp.s32 %0, 1, 0, p;\n}"
        : "=r"(r) : "d"(q[0]), "d"(q[1]), "d"(q[2]), "d"(q[3]), "d"(q[4]), "d"(q[5]), "d"(q[6]), "d"(q[7]), "d"(b));
    return r != 0;
}
__device__ __forceinline__ bool any_le4(const double* q, double b) {
    int r;
    asm("{\n.reg .pred p;\n"
        "setp.le.f64 p, %1, %5;\n setp.le.or.f64 p, %2, %5, p;\n setp.le.or.f64 p, %3, %5, p;\n setp.le.or.f64 p, %4, %5, p;\n"
        "selp.s32 %0, 1, 0, p;\n}"
        : "=r"(r) : "d"(q[0]), "d"(q[1]), "d"(q[2]), "d"(q[3]), "d"(b));
    return r != 0;
}
__device__ __forceinline__ bool any_le2(const double* q, double b) {
    int r;
    asm("{\n.reg .pred p;\n setp.le.f64 p, %1, %3;\n setp.le.or.f64 p, %2, %3, p;\n selp.s32 %0, 1, 0, p;\n}"
        : "=r"(r) : "d"(q[0]), "d"(q[1]), "d"(b));
    return r != 0;
}

__device__ __forceinline__ void eval_ss(const double* sm, const RowData* rd, double cm2, double cS0, double cS1, int cP0,
                                        int cP1, double delta, double& bq, double& bqd, unsigned long long& bk) {
    static_assert(RPG == 4, "any_le helpers are written for 4 rows per group");
    double q[2 * RPG];
#pragma unroll
    for (int u = 0; u < RPG; ++u) {
        const double2 e = lds2(sm + u * BOX_W);
        const double nS = -rd[u].S;
        q[2 * u] = __fma_rn(cm2, e.x, nS) - cS0;
        q[2 * u + 1] = __fma_rn(cm2, e.y, nS) - cS1;
    }
    if (any_le8(q, bqd)) {
#pragma unroll
        for (int u = 0; u < RPG; ++u) {
            const double2 e = lds2(sm + u * BOX_W);
            exact1(e.x, rd[u], cm2, cS0, cP0, bq, bk);
            exact1(e.y, rd[u], cm2, cS1, cP1, bq, bk);
        }
        bqd = bq + delta;
    }
}

__device__ __forceinline__ void eval_sp(const double* sm, const RowData* rd, double cm2, double cS0, int cP0, double delta,
                                        double& bq, double& bqd, unsigned long long& bk) {
    double q[RPG];
    const double h = cm2 * 0.5;
#pragma unroll
    for (int u = 0; u < RPG; ++u) {
        const double2 e = lds2(sm + u * BOX_W);
        q[u] = __fma_rn(h, e.x + e.y, -rd[u].S) - cS0;
    }
    if (any_le4(q, bqd)) {
#pragma unroll
        for (int u = 0; u < RPG; ++u) {
            const double2 e = lds2(sm + u * BOX_W);
            exact1((e.x + e.y) * 0.5, rd[u], cm2, cS0, cP0, bq, bk);
        }
        bqd = bq + delta;
    }
}

__device__ __forceinline__ void eval_pp(const double* sm, const RowData* rd, double cm2, double cS0, int cP0, double delta,
                                        double& bq, double& bqd, unsigned long long& bk) {
    double q[RPG / 2];
    const double h = cm2 * 0.25;
#pragma unroll
    for (int u = 0; u < RPG; u += 2) {
        const double2 e0 = lds2(sm + u * BOX_W);
        const double2 e1 = lds2(sm + (u + 1) * BOX_W);
        q[u / 2] = __fma_rn(h, (e0.x + e0.y) + (e1.x + e1.y), -rd[u].S) - cS0;
    }
    if (any_le2(q, bqd)) {
#pragma unroll
        for (int u = 0; u < RPG; u += 2)
            exact_pp(lds2(sm + u * BOX_W), lds2(sm + (u + 1) * BOX_W), rd[u], cm2, cS0, cP0, bq, bk);
        bqd = bq + delta;
    }
}

__global__ void __launch_bounds__(THREADS, 1)
k_scan_tma(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_row, const double* __restrict__ Sx,
           const int* __restrict__ pos, const unsigned long long* __restrict__ tile_mask, DevState* st, Partial* partials,
           const PeerTable* peers) {
    if (st->done || (st->mode != 0 && st->m > st->fallback)) return;   // NetMakerOriginal.java:361-366
    extern __shared__ __align__(1024) unsigned char smem[];
    // keep the ring pointer in the shared window (no generic-address loads): offset, not integer cast
    double* ring = reinterpret_cast<double*>(smem + ((1024u - (smem_u32(smem) & 1023u)) & 1023u));
    __shared__ uint64_t full_bar[STAGES], empty_bar[STAGES];
    __shared__ RowData rowdata[2][2][TILE_ROWS];   // [tile parity][box][row]: S = -inf where the row segment is not fetched
    __shared__ Partial wbest[THREADS / 32];
    __shared__ bool amLast;

    const int m = st->m, P2 = st->P2;
    const double cm2 = (double)st->c - 2.0;
    const int tid = threadIdx.x;
    const int ew = effective_world(st->world, m);   // ranks that share this scan (1: every rank scans all tiles)
    // the cluster created by the previous iteration: its u.Sx is still being summed by k_chain on a forked
    // branch, which also evaluates that cluster's pairs exactly; here its Sx reads as -inf, i.e. Q = +inf
    const int msk = st->mask_su;
    // k_prune's survivor masks (one 64-bit word per tile: bit 16*chunk + 8*box + row) when it pruned this launch, else all ones
    const bool pruned = st->prune_on;
    const int tfirst = (ew > 1 ? st->rank : 0) + ew * blockIdx.x, tstride = ew * gridDim.x;
    const long long ttotal = TileIter(m, 0, 1).total;
    const int lane = tid & 31;

    if (tid == 0) {
        if (blockIdx.x == 0) tl_stamp(st, TL_SCAN0);
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], CONSUMERS / 32); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    double bq = INFINITY;
    unsigned long long bk = ~0ull;
    // filter slack: bounds the rounding difference between the role-free q~ and the exact q.  Every rounding is
    // fl(x) = x(1+e) + h with |e| <= 2^-53 and |h| <= 2^-1075, h != 0 only for a product (or fma) whose result is below
    // 2^-1022 (a sum or difference that lands there is exact).  The relative parts give the first term: every value is
    // <= (c-2)*max|D| + 2c*max|D| and passes through <= 6 roundings in either form.  The absolute parts: the reference
    // rounds Dpq (the *0.5 / *0.25 of a pair mean; its error is then multiplied by c-2) and (c-2)*Dpq, the role-free
    // form rounds its fma once, and the product below may lose one more on underflow: <= (c+1) * 2^-1075, which
    // (c+2) * 2^-1074 covers twice over.  For distances in the normal range that term is far below one ulp of delta
    // and changes nothing.
    const double delta = 16.0 * 1.1102230246251565e-16 * (3.0 * (double)st->c + 2.0) * st->Dmax
                       + ((double)st->c + 2.0) * 4.9406564584124654e-324;
    double bqd = INFINITY;

    if (tid >= CONSUMERS) {
        // ===================== producer warp: issues the TMA loads of every chunk that holds a surviving row segment
        // A chunk whose 16 row segments all survive is fetched as the two 8 x 256 boxes; otherwise each surviving segment is
        // one 1 x 256 box (a pair row is two of them), and a chunk without survivors takes no stage at all.
        int stage = 0;
        uint32_t phase = 0;
        for (long long w = tfirst; w < ttotal; w += 32LL * tstride) {
            const long long tl = w + (long long)lane * tstride;
            const unsigned long long mk = tl < ttotal ? (pruned ? tile_mask[tl] : ~0ull) : 0ull;
            for (unsigned live = __ballot_sync(0xffffffffu, mk != 0); live; live &= live - 1) {
                const int src = __ffs(live) - 1;
                const unsigned long long tm = __shfl_sync(0xffffffffu, mk, src);
                int r0, cb0;
                TileIter(m, (int)(w + (long long)src * tstride), 1).decode(r0, cb0);
                const int rEnd = min(r0 + TILE_ROWS, m);
                for (int ch = 0, rc = r0; rc < rEnd; ++ch, rc += BOX_R) {
                    const unsigned cm = (unsigned)(tm >> (16 * ch)) & 0xffffu;
                    if (!cm) continue;
                    const int rcEnd = min(rc + BOX_R, rEnd);
                    double* dst = ring + (size_t)stage * (STAGE_BYTES / 8);
                    if (lane == 0) mbar_wait(&empty_bar[stage], phase ^ 1);
                    if (cm == 0xffffu) {
                        if (lane == 0) {
                            const bool second = (cb0 + BOX_W < rcEnd - 1) && (cb0 + BOX_W < m);
                            mbar_expect_tx(&full_bar[stage], second ? STAGE_BYTES : STAGE_BYTES / 2);
                            tma_load_2d(dst, &tmap, cb0, rc, &full_bar[stage]);
                            if (second) tma_load_2d(dst + BOX_R * BOX_W, &tmap, cb0 + BOX_W, rc, &full_bar[stage]);
                        }
                    } else {
                        if (lane == 0) mbar_expect_tx(&full_bar[stage], (uint32_t)__popc(cm) * (BOX_W * 8));
                        __syncwarp();
                        if (lane < 2 * BOX_R && ((cm >> lane) & 1u)) {
                            const int bx = lane / BOX_R, u = lane % BOX_R;
                            tma_load_2d(dst + bx * (BOX_R * BOX_W) + u * BOX_W, &tmap_row, cb0 + bx * BOX_W, rc + u, &full_bar[stage]);
                        }
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else {
        // ===================== consumer warps =====================
        int stage = 0;
        uint32_t phase = 0;
        const int grp = tid / GROUP, gt = tid % GROUP;
        const int box = gt >> 7, lc = (gt & 127) * 2;   // which box of the stage, local column
        const int uo = grp * RPG;                       // first chunk row of this group
        int tileParity = 0;
        for (long long w = tfirst; w < ttotal; w += 32LL * tstride) {   // the producer's tile sequence and masks
          const long long tl = w + (long long)lane * tstride;
          const unsigned long long mk = tl < ttotal ? (pruned ? tile_mask[tl] : ~0ull) : 0ull;
          for (unsigned live = __ballot_sync(0xffffffffu, mk != 0); live; live &= live - 1, tileParity ^= 1) {
            const int src = __ffs(live) - 1;
            const unsigned long long tm = __shfl_sync(0xffffffffu, mk, src);
            int r0, cb0;
            TileIter(m, (int)(w + (long long)src * tstride), 1).decode(r0, cb0);
            const int rEnd = min(r0 + TILE_ROWS, m);
            if (tid < 2 * TILE_ROWS && r0 + (tid % TILE_ROWS) < m) {   // stage the tile's row data, per box
                const int bx = tid / TILE_ROWS, i = tid % TILE_ROWS, r = r0 + i;
                const bool fetched = (tm >> (16 * (i / BOX_R) + BOX_R * bx + i % BOX_R)) & 1ull;
                rowdata[tileParity][bx][i].S = ((r & ~1) == msk || !fetched) ? -INFINITY : Sx[r];
                rowdata[tileParity][bx][i].pos = pos[r];
            }
            const int c0 = cb0 + box * BOX_W + lc;
            const bool cvalid = (c0 < m) && (c0 < rEnd - 1);   // some row of the tile lies strictly below column c0
            const bool colPair = c0 < P2;
            double cS0 = 0.0, cS1 = 0.0;
            int cP0 = 0, cP1 = 0;
            if (cvalid) {
                cS0 = Sx[c0]; cP0 = pos[c0];
                if (c0 + 1 < m) { cS1 = Sx[c0 + 1]; cP1 = pos[c0 + 1]; }
                if (c0 == msk) { cS0 = -INFINITY; cS1 = -INFINITY; }   // c0 is even, a masked pair is one thread's columns
            }
            asm volatile("bar.sync 1, %0;" ::"n"(CONSUMERS) : "memory");

            for (int ch = 0, rc = r0; rc < rEnd; ++ch, rc += BOX_R) {
                if (!((tm >> (16 * ch)) & 0xffffull)) continue;   // no surviving row segment: nothing was fetched
                const int rcEnd = min(rc + BOX_R, rEnd);
                mbar_wait(&full_bar[stage], phase);
                const double* sm = ring + (size_t)stage * (STAGE_BYTES / 8) + box * (BOX_R * BOX_W) + lc + uo * BOX_W;
                const int ra = rc + uo, rb = min(ra + RPG, rcEnd);   // this group's rows of the chunk
                const RowData* rd = &rowdata[tileParity][box][ra - r0];
                if (cvalid && c0 < rb - 1) {
                    const bool full_rows = (rcEnd - rc == BOX_R);
                    if (colPair && full_rows && rcEnd <= P2 && c0 < ra) {
                        // ---- pair rows x pair column, interior
                        eval_pp(sm, rd, cm2, cS0, cP0, delta, bq, bqd, bk);
                    } else if (colPair && full_rows && rc >= P2) {
                        // ---- single rows x pair column (always below the diagonal)
                        eval_sp(sm, rd, cm2, cS0, cP0, delta, bq, bqd, bk);
                    } else if (!colPair && full_rows && rc >= P2 && c0 + 1 < ra && c0 + 1 < m) {
                        // ---- single rows x two single columns, interior
                        eval_ss(sm, rd, cm2, cS0, cS1, cP0, cP1, delta, bq, bqd, bk);
                    } else if (colPair) {
                        // ---- generic pair column (diagonal / region boundary / ragged end)
                        for (int rr = ra; rr < rb;) {
                            const RowData r = rd[rr - ra];
                            const int rp = (int)r.pos;
                            const bool rowP = rp > cP0;
                            const double s1 = rowP ? r.S : cS0;
                            const double s2 = rowP ? cS0 : r.S;
                            if (rr < P2) {
                                if (c0 < rr) {
                                    const double2 e0 = lds2(sm + (rr - ra) * BOX_W);
                                    const double2 e1 = lds2(sm + (rr - ra + 1) * BOX_W);
                                    const double t1 = rowP ? e0.y : e1.x;
                                    const double t2 = rowP ? e1.x : e0.y;
                                    const double dpq = (((e0.x + t1) + t2) + e1.y) * 0.25;
                                    const double q = (cm2 * dpq - s1) - s2;
                                    FNN_CONSIDER(q, rp, cP0, rowP)
                                }
                                rr += 2;
                            } else {
                                const double2 e = lds2(sm + (rr - ra) * BOX_W);
                                const double dpq = (e.x + e.y) * 0.5;
                                const double q = (cm2 * dpq - s1) - s2;
                                FNN_CONSIDER(q, rp, cP0, rowP)
                                rr += 1;
                            }
                        }
                    } else {
                        // ---- generic single columns
                        for (int rr = max(max(ra, P2), c0 + 1); rr < rb; ++rr) {
                            const double2 e = lds2(sm + (rr - ra) * BOX_W);
                            const RowData r = rd[rr - ra];
                            const int rp = (int)r.pos;
                            {
                                const bool rowP = rp > cP0;
                                const double q = (cm2 * e.x - (rowP ? r.S : cS0)) - (rowP ? cS0 : r.S);
                                FNN_CONSIDER(q, rp, cP0, rowP)
                            }
                            if (c0 + 1 < rr) {
                                const bool rowP = rp > cP1;
                                const double q = (cm2 * e.y - (rowP ? r.S : cS1)) - (rowP ? cS1 : r.S);
                                FNN_CONSIDER(q, rp, cP1, rowP)
                            }
                        }
                    }
                }
                bqd = bq + delta;
                __syncwarp();
                if ((tid & 31) == 0) mbar_arrive(&empty_bar[stage]);
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
          }
        }
    }

    // ---- block min-loc, then the last block to finish reduces the per-block partials
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        double oq = __shfl_down_sync(0xffffffffu, bq, off);
        unsigned long long ok = __shfl_down_sync(0xffffffffu, bk, off);
        if (better(oq, ok, bq, bk)) { bq = oq; bk = ok; }
    }
    if ((tid & 31) == 0) wbest[tid >> 5] = Partial{bq, bk};
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < THREADS / 32; ++w)
            if (better(wbest[w].q, wbest[w].key, bq, bk)) { bq = wbest[w].q; bk = wbest[w].key; }
        partials[blockIdx.x] = Partial{bq, bk};
        __threadfence();
        unsigned int tk = atomicAdd(&st->ticket, 1u);
        amLast = (tk == gridDim.x - 1);
    }
    __syncthreads();
    if (amLast) {
        __threadfence();
        bq = INFINITY; bk = ~0ull;
        for (int b = tid; b < (int)gridDim.x; b += THREADS) {
            const double pq = __ldcg(&partials[b].q);
            const unsigned long long pk = __ldcg(&partials[b].key);
            if (better(pq, pk, bq, bk)) { bq = pq; bk = pk; }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            double oq = __shfl_down_sync(0xffffffffu, bq, off);
            unsigned long long ok = __shfl_down_sync(0xffffffffu, bk, off);
            if (better(oq, ok, bq, bk)) { bq = oq; bk = ok; }
        }
        __syncthreads();
        if ((tid & 31) == 0) wbest[tid >> 5] = Partial{bq, bk};
        __syncthreads();
        if (tid == 0) {
            for (int w = 1; w < THREADS / 32; ++w)
                if (better(wbest[w].q, wbest[w].key, bq, bk)) { bq = wbest[w].q; bk = wbest[w].key; }
            st->ticket = 0;
            tl_stamp(st, TL_SCAN1);
            if (ew > 1) {
                // post this rank's partial into every rank's mailbox (own included); every block of k_rx_stage merges.
                // Payloads first, ONE system-scope fence, then the tags.
                const int par = st->iter & 1;
                const long long tag = st->run_tag + (long long)st->iter + 1;
                for (int r = 0; r < st->world; ++r) mail_store_payload(&peers->box[r]->slot[par][st->rank], bq, bk);
                __threadfence_system();
                for (int r = 0; r < st->world; ++r) mail_store_tag(&peers->box[r]->slot[par][st->rank], tag);
            } else {
                // merged with k_patch's partial (the masked cluster) and decoded by k_rx_stage
                st->scanQ = bq;
                st->scanKey = bk;
            }
        }
    }
}

}  // namespace tma
