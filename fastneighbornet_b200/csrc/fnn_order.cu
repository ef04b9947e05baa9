// fnn_order.cu — B200-native Neighbor-Net ordering engine (seam B1 of include/fastnn.h).
//
// What the reference does (NetMakerOriginal.java:129-162): n-1 agglomeration iterations of
//   select (Q-criterion argmin over cluster pairs, :197-236 / NeighborNetCanonical.java:150-179)
//   -> pick node pair among <=4 (ComputeRx, :397-452) -> subtract sweep (:455-461, :681-696)
//   -> 2/3/4-way reduction with in-place D update (:570-726) -> add sweep (:517-536),
// then the circular-order expansion (:246-325).
//
// How this file does it (B200-first, not a translation):
//   * The whole agglomeration state lives in HBM and the loop runs device-side: five kernels on the
//     critical path of an iteration (scan, k_rx_stage, k_pick, k_rows, k_scatter) plus two on a forked
//     graph branch (k_chain + k_patch, overlapped with the NEXT iteration's scan), no host round trip,
//     replayed as a CUDA graph.  The host only expands the amalgamation log at the end (expandNodes
//     stays on the host, SURVEY §8 a13).
//   * Physical layout != reference layout.  The live nodes occupy matrix slots [0,m):
//     slots [0,P2) hold the paired clusters as aligned (rep, non-rep) slot pairs, slots
//     [P2,m) hold the singletons.  Every cluster pair's 1/2/4 cross entries are then one or
//     two aligned 16-byte loads, the selection scan is a dense coalesced stream over the
//     lower triangle (each cross-cluster entry read exactly once = the algorithmic bytes of
//     SURVEY §8d), and the matrix never fragments (SURVEY H4).  Keeping that layout costs
//     O(1) row/column moves (<=6 slots) per iteration.
//   * The reference's scan order is carried as data: pos[slot] is the node's index in the
//     Java netNodes[] array; the fused min-loc reduces on the key (Q, i, j) = (value, higher
//     position, lower position), which is exactly "first strict minimum in (i, j<i) order".
//   * Bit-exactness: compiled with --fmad=false.  u.Sx (a persistent left-to-right sum, :530-535) is
//     reproduced bit for bit by the verified binade-collapsed summation of fnn_exact_sum.cuh, OFF the
//     critical path: the next scan runs with the new cluster masked (Sx = -inf) while k_chain + k_patch
//     finishes u.Sx and evaluates the new cluster's 2 rows exactly; the two partial min-locs are merged by
//     whichever finishes last.  The <=4 ComputeRx sums (:549-561) only feed the 4-candidate pick, so a
//     parallel sum with a rigorous rounding bound decides it whenever the candidates are separated by
//     more than the bound (certified pick); otherwise, and always when a trace is recorded, the exact
//     left-to-right sums decide.
//
// No CPU fallback: every entry point fails with FNN_E_NODEVICE when there is no GPU.
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <string>
#include <vector>
#include <algorithm>
#include "fastnn.h"
#include "fnn_common.h"
#include "fnn_relaxed_sm.h"
#include "fnn_record.h"

namespace {

constexpr int MAXK = 8;         // changed slots per iteration (<= 6 used)
constexpr int SRC_NEW_U = -1;   // content marker: the new node u / v of this iteration
constexpr int SRC_NEW_V = -2;

struct DevState {
    // committed state
    int m, c, P2, num_nodes;
    int iter, done, n_amalg, skip;
    int error;                    // non-zero: a device-side strategy kernel gave up (pool overflow, no pair found)
    // selection result (k_scan)
    double selQ;
    int sel_i, sel_j;
    unsigned int ticket;
    int pad0;
    // event descriptor (k_pick)
    int kind;                     // 2, 3, 4; 5 = the 4-active/2-cluster special case
    int m_new, c_new, P2_new;
    int fX, fY, fZ, fW;           // formula rows: 3-way (X,Y,Z); 4-way (x2,x,y,y2)
    int sx, sxn, sy, syn;         // chosen x, x.nbr, y, y.nbr (old slots; -1 = none)
    int su;                       // base slot of the new cluster (new layout)
    int K;
    double Duv;                   // the order-dependent u-v entry (SURVEY F12)
    int chg_slot[MAXK];
    int chg_src[MAXK];
    double chg_Sx[MAXK];
    int final3[4];
    // mode-specific selection (Relaxed: written by k_relaxed_select; Random: by k_random_eval)
    int mode, mult, fallback, cx_pos, cy_pos;
    int rank, world;
    long long run_tag;            // (run counter << 32): makes mailbox tags unique across runs of one context
    int pick_x_id, pick_y_id, pick_kind;
    int cx, cxn, cy, cyn, need_rx;   // k_rx_stage: chosen clusters (slots) and whether ComputeRx is needed
    unsigned long long rng;       // java.util.Random state (48 bits)
    double Dmax;                  // max |D| at load time (slack of the scan's filter, fnn_scan_tma.cuh)
    double alg_bytes;             // running sum of the selection scan's algorithmic bytes (SURVEY §8d)
    // ---- chain off the critical path: the cluster created by the previous iteration is masked in the scan
    int mask_su;                  // base slot of the cluster whose u.Sx is still being summed (-1: none)
    unsigned int patch_ticket;    // k_patch: the last block to finish reduces the blocks' partial min-locs
    unsigned int commit_ticket;   // k_scatter: the last block to finish commits (m, c, P2, iter, done)
    int pad1;
    double scanQ, patchQ;         // partial min-locs: the masked scan / the new cluster's rows
    unsigned long long scanKey, patchKey;
    // ---- certified pick
    long long cert_ok, cert_fail; // picks decided by the bounded parallel sums / by the exact chains
    // ---- algorithmic bytes of the Relaxed row scans (K7) / Random samples (K9), SURVEY §8(d)
    unsigned long long strat_bytes;
    unsigned long long strat_units;   // row scans / samples
    // ---- optional in-graph timeline (env FNN_TIMELINE=iter0,count,file): globaltimer stamps of the kernels of a window of
    // iterations, the only way to see the real overlap and gaps inside a graph replay
    unsigned long long* tl;
    int tl_iter0, tl_count;
};
constexpr int TL_EVENTS = 16;
enum { TL_SCAN0 = 0, TL_SCAN1, TL_RX0, TL_RX1, TL_PICK0, TL_PICK1, TL_ROWS0, TL_ROWS1, TL_SCAT0, TL_SCAT1, TL_CHAIN0, TL_CHAIN1,
       TL_PATCH1, TL_SEL0, TL_SEL1 };

constexpr int RX_BLOCKS_MAX = 1024;   // per-block partial ComputeRx sums: [block][8] = 4 sums + 4 sums of |terms|

struct Partial { double q; unsigned long long key; };


// Multi-GPU selection exchange (SURVEY §8e): every rank scans 1/world of the tiles and posts its partial
// (Q, i, j) min-loc into slot [iteration parity][rank] of EVERY peer's mailbox with plain stores over
// NVLink (peer memory mapped through CUDA IPC); the tag carries the iteration number.
constexpr int MAX_WORLD = 8;
// below this many active nodes a full scan costs less than the cross-GPU exchange: every rank scans everything itself
constexpr int SHARD_MIN_ACTIVE = 4096;
__device__ __forceinline__ int effective_world(int world, int m) { return m > SHARD_MIN_ACTIVE ? world : 1; }
// payload first, then a system-scope fence, then the tag (release); the reader spins on the tag (acquire) and only then
// reads the payload - no reliance on a 16-byte store being single-copy atomic across NVLink
struct __align__(32) MailSlot { double q; unsigned long long key; long long tag; long long pad; };
__device__ __forceinline__ void mail_store_payload(MailSlot* ms, double q, unsigned long long key) {
    asm volatile("st.volatile.global.f64 [%0], %1;" ::"l"(&ms->q), "d"(q) : "memory");
    asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(&ms->key), "l"(key) : "memory");
}
__device__ __forceinline__ void mail_store_tag(MailSlot* ms, long long tag) {   // after a __threadfence_system()
    asm volatile("st.relaxed.sys.global.s64 [%0], %1;" ::"l"(&ms->tag), "l"(tag) : "memory");
}
__device__ __forceinline__ long long mail_load_tag(const MailSlot* ms) {
    long long t;
    asm volatile("ld.acquire.sys.global.s64 %0, [%1];" : "=l"(t) : "l"(&ms->tag) : "memory");
    return t;
}
__device__ __forceinline__ void mail_load_payload(const MailSlot* ms, double& q, unsigned long long& key) {
    asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(q) : "l"(&ms->q) : "memory");
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(key) : "l"(&ms->key) : "memory");
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
constexpr unsigned long long MAIL_TIMEOUT_NS = 30ull * 1000000000ull;   // a peer that never posts: give up, do not hang
__device__ __forceinline__ void tl_stamp(DevState* st, int ev) {
    unsigned long long* tl = st->tl;
    if (tl) {
        const int k = st->iter - st->tl_iter0;
        if (k >= 0 && k < st->tl_count) tl[k * TL_EVENTS + ev] = global_ns();
    }
}
struct Mailbox { MailSlot slot[2][MAX_WORLD]; };
struct PeerTable { Mailbox* box[MAX_WORLD]; };

#define TWO_THIRDS (2.0 / 3.0)

__device__ __forceinline__ bool better(double q, unsigned long long k, double bq, unsigned long long bk) {
    return (q < bq) || (q == bq && k < bk);
}

}  // namespace
#include <cuda.h>
namespace {
#include "fnn_scan_tma.cuh"
#include "fnn_exact_sum.cuh"
#include "fnn_modes.cuh"

// ------------------------------------------------------------------ init kernels
__global__ void k_init_nodes(int n, int* id, int* pos, int* p2s, DevState* st, int mode, int mult, int fallback, long long seed,
                             int rank, int world, long long run_tag, unsigned long long* tl, int tl_iter0, int tl_count) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) { id[t] = t + 1; pos[t] = t; p2s[t] = t; }
    if (t == 0) {
        memset(st, 0, sizeof(DevState));
        st->m = n; st->c = n; st->P2 = 0; st->num_nodes = n;
        st->mode = mode; st->mult = mult; st->fallback = fallback;
        st->rank = rank; st->world = world; st->run_tag = run_tag;
        st->rng = ((unsigned long long)seed ^ 0x5DEECE66DULL) & ((1ULL << 48) - 1);   // java.util.Random(seed)
        st->mask_su = -1;
        st->patchQ = INFINITY; st->patchKey = ~0ull;
        st->scanQ = INFINITY; st->scanKey = ~0ull;
        st->tl = tl; st->tl_iter0 = tl_iter0; st->tl_count = tl_count;
    }
}

// K1: Sx[k] = sum_{j != k} D[k][j], ascending j (NetMakerOriginal.java:164-191).  Thread k walks
// column k (== row k by symmetry) so that a warp reads 256 contiguous bytes per step.
__global__ void k_rowsum(const double* __restrict__ D, int64_t ld, int n, double* Sx, DevState* st) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    double s = 0.0, mx = 0.0;
    const double* col = D + k;
#pragma unroll 8
    for (int j = 0; j < n; ++j) {
        double v = col[(int64_t)j * ld];
        if (j != k) { s += v; mx = fmax(mx, fabs(v)); }
    }
    Sx[k] = s;
    // non-negative doubles order like their bit patterns
    if (st) atomicMax(reinterpret_cast<unsigned long long*>(&st->Dmax), (unsigned long long)__double_as_longlong(mx));
}

__global__ void k_zero_diag(double* D, int64_t ld, int n) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) D[(int64_t)k * ld + k] = 0.0;
}

// ------------------------------------------------------------------ sequential chains
// Sum NR rows of length len strictly left to right (the reference's accumulation order).
// All threads stage tiles into shared memory through `load(row, i)`; lane r of warp 0 owns
// chain r.  Double-buffered so the staging of tile k+1 overlaps the dependent adds of tile k.
constexpr int CH_TILE = 1024;
constexpr size_t PICK_SMEM = sizeof(xsum::Smem) > 2 * 4 * CH_TILE * sizeof(double) ? sizeof(xsum::Smem) : 2 * 4 * CH_TILE * sizeof(double);
// k_chain + k_patch: one chain.  When it fits, the whole staged chain is first copied into shared memory with every load in
// flight at once (one L2 round trip instead of one per pass / per opened segment of the exact summation).
constexpr size_t CHAIN_SMEM_BASE = sizeof(xsum::SmemN<1>) > 2 * CH_TILE * sizeof(double) ? sizeof(xsum::SmemN<1>) : 2 * CH_TILE * sizeof(double);
constexpr size_t CHAIN_SMEM_MAX = 220 * 1024;

template <int NR, typename Loader>
__device__ void block_seq_sum(double (*buf)[NR][CH_TILE], int len, Loader load, double* out /*[NR]*/) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const int ntiles = (len + CH_TILE - 1) / CH_TILE;
    double acc = 0.0;
    // prologue: tile 0
    for (int e = tid; e < NR * CH_TILE; e += nt) {
        int r = e / CH_TILE, i = e % CH_TILE;
        buf[0][r][i] = (i < len) ? load(r, i) : 0.0;
    }
    __syncthreads();
    for (int t = 0; t < ntiles; ++t) {
        const int cur = t & 1;
        if (tid >= 32) {
            if (t + 1 < ntiles) {
                const int b0 = (t + 1) * CH_TILE;
                for (int e = tid - 32; e < NR * CH_TILE; e += nt - 32) {
                    int r = e / CH_TILE, i = e % CH_TILE;
                    buf[cur ^ 1][r][i] = (b0 + i < len) ? load(r, b0 + i) : 0.0;
                }
            }
        } else if (tid < NR) {
            const int cnt = min(CH_TILE, len - t * CH_TILE);
            const double* row = buf[cur][tid];
            int i = 0;
            for (; i + 8 <= cnt; i += 8) {
                double v0 = row[i], v1 = row[i + 1], v2 = row[i + 2], v3 = row[i + 3];
                double v4 = row[i + 4], v5 = row[i + 5], v6 = row[i + 6], v7 = row[i + 7];
                acc += v0; acc += v1; acc += v2; acc += v3; acc += v4; acc += v5; acc += v6; acc += v7;
            }
            for (; i < cnt; ++i) acc += row[i];
        }
        __syncthreads();
    }
    if (tid < NR) out[tid] = acc;
    __syncthreads();
}

__device__ __forceinline__ int nbr_of(int s, int P2) { return s < P2 ? (s ^ 1) : -1; }

// reference netNodes[y.pos] = netNodes[num_active-1] (NetMakerOriginal.java:641-643) on the
// position attributes; posU/posV are the not-yet-placed new nodes.
__device__ void remove_pos(int* pos, int* p2s, int m_cur, int yp, int& posU, int& posV) {
    const int last = m_cur - 1;
    if (yp == last) return;
    if (posU == last) posU = yp;
    else if (posV == last) posV = yp;
    else { int L = p2s[last]; pos[L] = yp; p2s[yp] = L; }
}

// the order-dependent D[u][v] of agg3way (NetMakerOriginal.java:653-657, SURVEY F12)
__device__ __forceinline__ double duv_rule(bool uFirst, double dZX, double dYX, double dYZ) {
    if (uFirst) { double A = TWO_THIRDS * dZX + dYX / 3.0; return TWO_THIRDS * A + dYZ / 3.0; }
    double B = TWO_THIRDS * dZX + dYZ / 3.0;
    return TWO_THIRDS * B + dYX / 3.0;
}

// ------------------------------------------------------------------ K3a: selection result -> clusters
// Computed redundantly by one thread of EVERY block of k_rx_stage (a handful of dependent L2 loads), so that it costs no
// launch, no ticket and no fence: merge the partial min-locs - the masked scan's (single GPU) or every rank's, posted
// into this rank's mailbox over NVLink (multi-GPU) - with k_chain + k_patch's partial for the masked cluster; then Cx, Cy from
// the (i, j) key (or from the Relaxed/Random strategy) and the id-order swap of NetMakerOriginal.java:376-380.
struct Sel { int cx, cxn, cy, cyn, need_rx, ok; double q; int i, j; };
__device__ Sel select_decode(const int* __restrict__ id, const int* __restrict__ p2s, const DevState* st, const Mailbox* mail) {
    Sel r{-1, -1, -1, -1, 0, 1, 0.0, 0, 0};
    const int m = st->m, P2 = st->P2;
    if (m == 4 && st->c == 2) return r;   // special case is handled by k_pick
    const bool strategy = (st->mode != 0 && m > st->fallback);
    int cx, cy;
    if (!strategy) {
        double bq = st->scanQ;
        unsigned long long bk = st->scanKey;
        if (effective_world(st->world, m) > 1) {
            const int par = st->iter & 1;
            bq = INFINITY; bk = ~0ull;
            const long long want = st->run_tag + (long long)st->iter + 1;   // posted by every rank's scan of this iteration
            const unsigned long long t_start = global_ns();
            for (int k = 0; k < st->world; ++k) {
                const MailSlot* ms = &mail->slot[par][k];
                unsigned spins = 0;
                while (mail_load_tag(ms) != want) {
                    if ((++spins & 0x3ff) == 0 && global_ns() - t_start > MAIL_TIMEOUT_NS) { r.ok = 0; return r; }   // a peer never posted
                }
                double q; unsigned long long key;
                mail_load_payload(ms, q, key);
                if (better(q, key, bq, bk)) { bq = q; bk = key; }
            }
        }
        // the cluster the scan had masked, evaluated exactly by k_chain + k_patch
        if (better(st->patchQ, st->patchKey, bq, bk)) { bq = st->patchQ; bk = st->patchKey; }
        r.q = bq; r.i = (int)(bk >> 32); r.j = (int)(bk & 0xffffffffu);
        cx = p2s[r.i]; cy = p2s[r.j];
    } else { cx = p2s[st->cx_pos]; cy = p2s[st->cy_pos]; }   // Relaxed: k_relaxed_select, Random: k_random_eval
    if (id[cx] > id[cy]) { const int t = cx; cx = cy; cy = t; }
    r.cx = cx; r.cxn = cx < P2 ? (cx ^ 1) : -1;
    r.cy = cy; r.cyn = cy < P2 ? (cy ^ 1) : -1;
    r.need_rx = (r.cxn >= 0 || r.cyn >= 0);
    return r;
}

// ------------------------------------------------------------------ K3b: ComputeRx operands on all SMs
// For the <=4 rows z in {Cx, Cx.nbr, Cy, Cy.nbr}: term_i = w_i * D[z][p_i], w = 1 for the four chosen nodes and singletons,
// 1/2 otherwise (NetMakerOriginal.java:555-558).  Two products:
//   * rx_part[block][0..3] = this block's share of sum_i term_i, [4..7] = of sum_i |term_i| (any order: they only feed the
//     certified pick of k_pick, which bounds the difference to the reference's left-to-right sum);
//   * rxs[r][k*1024 + t] = term of position i = t*L + k (segment-transposed, so the exact summation block reads coalesced).
__global__ void __launch_bounds__(256)
k_rx_stage(const double* __restrict__ D, int64_t ld, const int* __restrict__ id, const int* __restrict__ pos,
           const int* __restrict__ p2s, DevState* st, const Mailbox* mail, double* __restrict__ rxs, int64_t rxs_ld,
           double* __restrict__ rx_part) {
    if (st->done) return;
    __shared__ Sel sel;
    if (threadIdx.x == 0) {
        if (blockIdx.x == 0) tl_stamp(st, TL_SEL0);
        sel = select_decode(id, p2s, st, mail);
        if (blockIdx.x == 0) {   // publish for k_pick
            if (!sel.ok) { st->error = 30; st->done = 1; st->skip = 1; }   // a peer rank never posted: surface FNN_E_STATE
            const int m_ = st->m;
            const bool strategy = (st->mode != 0 && m_ > st->fallback);
            st->cx = sel.cx; st->cxn = sel.cxn; st->cy = sel.cy; st->cyn = sel.cyn; st->need_rx = sel.need_rx;
            if (!strategy && sel.cx >= 0) {
                st->selQ = sel.q; st->sel_i = sel.i; st->sel_j = sel.j;
                st->alg_bytes += 4.0 * (double)m_ * ((double)m_ - 1.0) - 4.0 * (double)st->P2 + 8.0 * (double)m_;
            }
            tl_stamp(st, TL_RX0);
        }
    }
    __syncthreads();
    if (!sel.ok || !sel.need_rx) return;
    const int m = st->m, P2 = st->P2;
    const int Cx = sel.cx, Cxn = sel.cxn, Cy = sel.cy, Cyn = sel.cyn;
    const int L = (m + xsum::THREADS - 1) / xsum::THREADS;
    const int zs[4] = {Cx, Cxn, Cy, Cyn};
    double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < m; s += gridDim.x * blockDim.x) {
        const int i = pos[s];
        const bool full = (s >= P2) || s == Cx || s == Cxn || s == Cy || s == Cyn;
        const int64_t dst = (int64_t)(i % L) * xsum::THREADS + (i / L);
#pragma unroll
        for (int r = 0; r < 4; ++r)
            if (zs[r] >= 0) {
                const double v = D[(int64_t)zs[r] * ld + s];
                const double t = full ? v : v * 0.5;
                rxs[(int64_t)r * rxs_ld + dst] = t;
                acc[r] += t;
                acc[4 + r] += fabs(t);
            }
    }
    __shared__ double wsum[8][8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        double v = acc[q];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5][q] = v;
    }
    __syncthreads();
    if (threadIdx.x < 8) {
        double v = 0.0;
        for (int w = 0; w < 8; ++w) v += wsum[w][threadIdx.x];
        rx_part[blockIdx.x * 8 + threadIdx.x] = v;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) tl_stamp(st, TL_RX1);
}

// ------------------------------------------------------------------ K3: pick + bookkeeping (one block)
constexpr int PICK_THREADS = 1024;

__global__ void __launch_bounds__(PICK_THREADS, 1)
k_pick(double* D, int64_t ld, double* Sx, int* id, int* pos, int* p2s, DevState* st, int* amalg, double* trace, int serial_chain,
       const double* __restrict__ rxs, int64_t rxs_ld, const double* __restrict__ rx_part, int rx_blocks, int force_exact) {
    extern __shared__ unsigned char smem_raw[];
    double (*buf)[4][CH_TILE] = reinterpret_cast<double (*)[4][CH_TILE]>(smem_raw);
    __shared__ double rx[4];
    __shared__ double rxa[8];
    __shared__ int s_exact, s_kstar;
    if (st->done) return;
    const int m = st->m, c = st->c, P2 = st->P2;
    const int tid = threadIdx.x;
    if (tid == 0) tl_stamp(st, TL_PICK0);

    // ---- special case: 4 active nodes in 2 clusters (NetMakerOriginal.java:343-360)
    if (m == 4 && c == 2) {
        if (tid == 0) {
            const int p = p2s[0], pn = p ^ 1;
            const int q = (p2s[1] != pn) ? p2s[1] : p2s[2];
            const int qn = q ^ 1;
            auto d = [&](int a, int b) { return D[(int64_t)a * ld + b]; };
            int X = p, Y, Z;
            if (d(p, q) + d(pn, qn) < d(p, qn) + d(pn, q)) { Y = q; Z = qn; } else { Y = qn; Z = q; }
            const int nn = st->num_nodes;
            int posU = pos[X], posV = pos[Z];
            remove_pos(pos, p2s, 4, pos[Y], posU, posV);
            int* lg = amalg + 5 * st->n_amalg;
            lg[0] = nn + 1; lg[1] = nn + 2; lg[2] = id[X]; lg[3] = id[Y]; lg[4] = id[Z];
            st->n_amalg += 1;
            st->num_nodes = nn + 2;
            st->final3[pos[pn]] = id[pn];
            st->final3[posU] = nn + 1;
            st->final3[posV] = nn + 2;
            if (trace) {
                double* tr = trace + 8 * (int64_t)st->iter;
                tr[0] = 4; tr[1] = 2; tr[2] = id[p]; tr[3] = id[q]; tr[4] = id[Y]; tr[5] = 0; tr[6] = 5; tr[7] = 0.0;
            }
            st->iter += 1;
            st->done = 1;
            st->skip = 1;
        }
        return;
    }

    const int Cx = st->cx, Cxn = st->cxn, Cy = st->cy, Cyn = st->cyn;   // k_rx_stage (select_decode)

    // ---- warm this SM's L1 with the O(1) scalars the single control thread is about to chase one after another
    // (the 4x4 distances among the chosen nodes, id/pos of the chosen and of the slots a layout move can touch)
    if (tid >= 32 && tid < 96) {
        const int k = tid - 32;
        const int zs4[4] = {Cx, Cxn, Cy, Cyn};
        const void* a = nullptr;
        if (k < 16) { const int r = zs4[k >> 2], q = zs4[k & 3]; if (r >= 0 && q >= 0) a = D + (int64_t)r * ld + q; }
        else if (k < 40) {
            const int j = (k - 16) >> 1;   // 0..11
            const int cand[12] = {Cx, Cxn, Cy, Cyn, m - 1, m - 2, P2 - 2, P2 - 1, P2, P2 + 1, m - 3, P2 - 4};
            const int sl = cand[j];
            if (sl >= 0 && sl < m) a = ((k & 1) ? (const void*)(pos + sl) : (const void*)(id + sl));
        } else if (k < 43) { const int q = m - 1 - (k - 40); if (q >= 0) a = p2s + q; }
        if (a) asm volatile("prefetch.global.L1 [%0];" ::"l"(a));
    }

    // ---- certified pick: the <=4 ComputeRx sums only decide which of the <=4 candidate pairs is joined (:428-452).
    // R~ = sum of k_rx_stage's per-block partials (some order), A = the same over |terms|.  Any two summation orders of
    // the same m terms differ by at most 2*gamma_m*A (gamma_m = m*u/(1-m*u), u = 2^-53), so with E = (2m+256)*u*A the
    // reference's left-to-right sum lies in [R~-E, R~+E]; each candidate Q = (f*d - Ra) - Rb then lies within
    // e = 1.01*(Ea+Eb) + 8u*(|f*d|+|Ra|+|Rb|) of its value computed from R~.  If the smallest candidate is separated
    // from every other one by more than the two bounds, the exact sums would pick the same pair: no chain needed.
    // Otherwise (near-ties, e.g. integer matrices), and whenever a trace is recorded (its `best` column is the exact
    // value, and the certified decision is then cross-checked against it), the exact sums decide.
    const bool need_rx = (Cxn >= 0 || Cyn >= 0);
    if (need_rx) {
        // the control thread's four candidate distances are requested before the reduction below, not after it
        double dcand[4] = {0.0, 0.0, 0.0, 0.0};
        if (tid == 0) {
            const int zs4[4] = {Cx, Cxn, Cy, Cyn};
            const int ra[4] = {0, 1, 0, 1}, rb[4] = {2, 2, 3, 3};
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (zs4[ra[k]] >= 0 && zs4[rb[k]] >= 0) dcand[k] = D[(int64_t)zs4[ra[k]] * ld + zs4[rb[k]]];
        }
        if (tid < 256) {   // warp w sums quantity w over the blocks
            const int q = tid >> 5, lane = tid & 31;
            double v = 0.0;
            for (int b = lane; b < rx_blocks; b += 32) v += rx_part[b * 8 + q];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
            if (lane == 0) rxa[q] = v;
        }
        __syncthreads();
        if (tid == 0) {
            const double U = 1.1102230246251565e-16;
            const double f = (double)(c + (Cxn >= 0) + (Cyn >= 0)) - 2.0;
            const int ra[4] = {0, 1, 0, 1}, rb[4] = {2, 2, 3, 3};
            double Q[4], e[4];
            bool pres[4] = {true, Cxn >= 0, Cyn >= 0, Cxn >= 0 && Cyn >= 0};
            bool finite = true;
            int ks = 0;
            for (int k = 0; k < 4; ++k) {
                if (!pres[k]) continue;
                const double Ra = rxa[ra[k]], Rb = rxa[rb[k]];
                const double Ea = rxa[4 + ra[k]] * ((2.0 * (double)m + 256.0) * U), Eb = rxa[4 + rb[k]] * ((2.0 * (double)m + 256.0) * U);
                const double t = f * dcand[k];
                Q[k] = (t - Ra) - Rb;
                e[k] = 1.01 * (Ea + Eb) + 8.0 * U * (fabs(t) + fabs(Ra) + fabs(Rb));
                finite = finite && isfinite(Q[k]) && isfinite(e[k]);
                if (Q[k] < Q[ks]) ks = k;
            }
            bool cert = finite;
            for (int k = 0; k < 4 && cert; ++k)
                if (pres[k] && k != ks && !(Q[ks] + e[ks] < Q[k] - e[k])) cert = false;
            s_kstar = cert ? ks : -1;
            s_exact = (!cert || force_exact || trace != nullptr) ? 1 : 0;
        }
        __syncthreads();
    }

    // ---- ComputeRx x<=4 (:413-420, :549-561): sequential in position order
    if (need_rx && s_exact) {
        const int zs[4] = {Cx, Cxn, Cy, Cyn};
        const int L = (m + xsum::THREADS - 1) / xsum::THREADS;   // rxs is segment-transposed by k_rx_stage
        auto load_seg = [&](int r, int t, int k) -> double { return rxs[(int64_t)r * rxs_ld + (int64_t)k * xsum::THREADS + t]; };
        auto load_lin = [&](int r, int i) -> double { return zs[r] < 0 ? 0.0 : load_seg(r, i / L, i % L); };
        if (serial_chain) block_seq_sum<4>(buf, m, load_lin, rx);
        else xsum::block_exact_seq_sum<4>(reinterpret_cast<xsum::Smem*>(smem_raw), m, load_seg, [&](int r) { return zs[r] >= 0; }, rx);
    } else {
        if (tid < 4) rx[tid] = 0.0;
        __syncthreads();
    }

    if (tid != 0) return;
    // ================= single-thread control: everything below is O(1) =================
    auto d = [&](int a, int b) { return D[(int64_t)a * ld + b]; };
    int x = Cx, y = Cy;
    if (need_rx && !s_exact) {
        // certified: candidate order (Cx,Cy), (Cx.nbr,Cy), (Cx,Cy.nbr), (Cx.nbr,Cy.nbr)
        const int ks = s_kstar;
        x = (ks & 1) ? Cxn : Cx;
        y = (ks & 2) ? Cyn : Cy;
        atomicAdd((unsigned long long*)&st->cert_ok, 1ull);   // result unused: no round trip
    } else {
        int mm = c + (Cxn >= 0) + (Cyn >= 0);
        const double f = (double)mm - 2.0;
        int kx = 0;
        double best = (f * d(Cx, Cy) - rx[0]) - rx[2];
        if (Cxn >= 0) { double q = (f * d(Cxn, Cy) - rx[1]) - rx[2]; if (q < best) { x = Cxn; y = Cy; best = q; kx = 1; } }
        if (Cyn >= 0) { double q = (f * d(Cx, Cyn) - rx[0]) - rx[3]; if (q < best) { x = Cx; y = Cyn; best = q; kx = 2; } }
        if (Cxn >= 0 && Cyn >= 0) { double q = (f * d(Cxn, Cyn) - rx[1]) - rx[3]; if (q < best) { x = Cxn; y = Cyn; best = q; kx = 3; } }
        if (need_rx) {
            if (s_kstar >= 0) {   // exact sums were computed although the pick was certifiable: cross-check the certificate
                atomicAdd((unsigned long long*)&st->cert_ok, 1ull);
                if (s_kstar != kx) { st->error = 21; st->done = 1; st->skip = 1; return; }
            } else atomicAdd((unsigned long long*)&st->cert_fail, 1ull);
        }
        if (trace) {
            double* tr = trace + 8 * (int64_t)st->iter;
            tr[0] = m; tr[1] = c; tr[2] = id[Cx]; tr[3] = id[Cy]; tr[4] = id[x]; tr[5] = id[y]; tr[7] = best;
        }
    }
    const int xn = nbr_of(x, P2), yn = nbr_of(y, P2);
    st->sx = x; st->sxn = xn; st->sy = y; st->syn = yn;
    st->pick_x_id = id[x]; st->pick_y_id = id[y];
    const int nn = st->num_nodes;
    int K = 0;
    int cslot[MAXK], csrc[MAXK], cid[MAXK], cpos[MAXK];
    auto add_old = [&](int slot, int src) { cslot[K] = slot; csrc[K] = src; cid[K] = id[src]; cpos[K] = pos[src]; ++K; };
    auto add_new = [&](int slot, int marker, int nid, int npos) { cslot[K] = slot; csrc[K] = marker; cid[K] = nid; cpos[K] = npos; ++K; };
    int kind;
    if (xn < 0 && yn < 0) {
        // ---------- 2-way (:462-464, :570-577): x (smaller id) becomes the representative
        kind = 2;
        const int T0 = P2, T1 = P2 + 1;
        add_old(T0, x);
        add_old(T1, y);
        int vac[2], nv = 0, dsp[2], ndp = 0;
        if (x != T0 && x != T1) vac[nv++] = x;
        if (y != T0 && y != T1) vac[nv++] = y;
        if (T0 != x && T0 != y) dsp[ndp++] = T0;
        if (T1 != x && T1 != y) dsp[ndp++] = T1;
        for (int i = 0; i < nv; ++i) add_old(vac[i], dsp[i]);
        st->m_new = m; st->c_new = c - 1; st->P2_new = P2 + 2; st->su = T0;
        st->fX = st->fY = st->fZ = st->fW = -1;
        st->Duv = 0.0;
    } else if (xn < 0 || yn < 0) {
        // ---------- 3-way (:465-482, :589-674): X isolated, (Y,Z) a pair
        kind = 3;
        const int X = (xn < 0) ? x : y;
        const int Y = (xn < 0) ? y : x;
        const int Z = Y ^ 1;
        int posU = pos[X], posV = pos[Z];
        const int idX = id[X], idY = id[Y], idZ = id[Z];
        remove_pos(pos, p2s, m, pos[Y], posU, posV);
        st->Duv = duv_rule(posU < posV, d(Z, X), d(Y, X), d(Y, Z));
        const int b = Y & ~1;
        add_new(b, SRC_NEW_U, nn + 1, posU);
        add_new(b + 1, SRC_NEW_V, nn + 2, posV);
        if (X != m - 1) add_old(X, m - 1);
        int* lg = amalg + 5 * st->n_amalg;
        lg[0] = nn + 1; lg[1] = nn + 2; lg[2] = idX; lg[3] = idY; lg[4] = idZ;
        st->n_amalg += 1;
        st->num_nodes = nn + 2;
        st->m_new = m - 1; st->c_new = c - 1; st->P2_new = P2; st->su = b;
        st->fX = X; st->fY = Y; st->fZ = Z; st->fW = -1;
    } else {
        // ---------- 4-way (:483-487, :707-726): agg3way(x2,x,y) then agg3way(u,u.nbr,y2)
        kind = 4;
        const int x2 = xn, y2 = yn;
        int posU = pos[x2], posV = pos[y];
        const int idx2 = id[x2], idx = id[x], idy = id[y], idy2 = id[y2];
        remove_pos(pos, p2s, m, pos[x], posU, posV);
        const double duv1 = duv_rule(posU < posV, d(y, x2), d(x, x2), d(x, y));
        const double u1y2 = TWO_THIRDS * d(x2, y2) + d(x, y2) / 3.0;
        const double v1y2 = TWO_THIRDS * d(y, y2) + d(x, y2) / 3.0;
        int posU2 = posU, posV2 = pos[y2];
        remove_pos(pos, p2s, m - 1, posV, posU2, posV2);
        st->Duv = duv_rule(posU2 < posV2, u1y2, duv1, v1y2);
        int* lg = amalg + 5 * st->n_amalg;
        lg[0] = nn + 1; lg[1] = nn + 2; lg[2] = idx2; lg[3] = idx; lg[4] = idy;
        lg[5] = nn + 3; lg[6] = nn + 4; lg[7] = nn + 1; lg[8] = nn + 2; lg[9] = idy2;
        st->n_amalg += 2;
        st->num_nodes = nn + 4;
        const int bx = x & ~1, by = y & ~1;
        const int A = min(bx, by), B = max(bx, by), Lp = P2 - 2;
        add_new(A, SRC_NEW_U, nn + 3, posU2);
        add_new(A + 1, SRC_NEW_V, nn + 4, posV2);
        if (B != Lp) { add_old(B, Lp); add_old(B + 1, Lp + 1); }
        const int S = m - P2;
        if (S >= 2) { add_old(Lp, m - 2); add_old(Lp + 1, m - 1); }
        else if (S == 1) { add_old(Lp, m - 1); }
        st->m_new = m - 2; st->c_new = c - 1; st->P2_new = P2 - 2; st->su = A;
        st->fX = x2; st->fY = x; st->fZ = y; st->fW = y2;
    }
    if (trace) trace[8 * (int64_t)st->iter + 6] = kind;
    st->kind = kind;
    st->pick_kind = kind;
    st->K = K;
    // publish the new layout's node tables (sources were captured above, so overlaps are safe)
    for (int k = 0; k < K; ++k) {
        st->chg_slot[k] = cslot[k];
        st->chg_src[k] = csrc[k];
        st->chg_Sx[k] = 0.0;
    }
    for (int k = 0; k < K; ++k) {
        id[cslot[k]] = cid[k];
        pos[cslot[k]] = cpos[k];
        p2s[cpos[k]] = cslot[k];
    }
    st->skip = 0;
    tl_stamp(st, TL_PICK1);
}

// formula rows of the new nodes at old column a (bystander columns; order independent)
struct Formula {
    int kind, X, Y, Z, W;
    __device__ __forceinline__ void eval(const double* D, int64_t ld, int a, double& fu, double& fv) const {
        if (kind == 3) {
            const double dx = D[(int64_t)X * ld + a], dy = D[(int64_t)Y * ld + a], dz = D[(int64_t)Z * ld + a];
            fu = TWO_THIRDS * dx + dy / 3.0;
            fv = TWO_THIRDS * dz + dy / 3.0;
        } else {  // 4-way: (x2, x, y, y2) = (X, Y, Z, W)
            const double dx2 = D[(int64_t)X * ld + a], dx = D[(int64_t)Y * ld + a];
            const double dy = D[(int64_t)Z * ld + a], dy2 = D[(int64_t)W * ld + a];
            const double u1 = TWO_THIRDS * dx2 + dx / 3.0;
            const double v1 = TWO_THIRDS * dy + dx / 3.0;
            fu = TWO_THIRDS * u1 + v1 / 3.0;
            fv = TWO_THIRDS * dy2 + v1 / 3.0;
        }
    }
};

// cluster distance D(p-cluster, x) in the subtract sweep's role order (:681-696): p the
// bystander representative (even slot if paired), x the chosen node, xn its neighbour or -1.
__device__ __forceinline__ double sub_dist(const double* D, int64_t ld, int p, bool pPair, int x, int xn) {
    const double* rx = D + (int64_t)x * ld;
    if (xn < 0) {
        if (!pPair) return rx[p];
        return (rx[p] + rx[p + 1]) * 0.5;
    }
    const double* rxn = D + (int64_t)xn * ld;
    if (!pPair) return (rx[p] + rxn[p]) * 0.5;
    return (((rx[p] + rxn[p]) + rx[p + 1]) + rxn[p + 1]) * 0.25;
}

// ------------------------------------------------------------------ K4+K5a: subtract sweep + build changed rows
__global__ void __launch_bounds__(256)
k_rows(const double* __restrict__ D, int64_t ld, double* Sx, DevState* st, double* scratch) {
    if (st->done || st->skip) return;
    if (blockIdx.x == 0 && threadIdx.x == 0) tl_stamp(st, TL_ROWS0);
    const int m = st->m, P2 = st->P2, m_new = st->m_new, K = st->K;
    __shared__ int cslot[MAXK], csrc[MAXK];
    if (threadIdx.x < MAXK) { cslot[threadIdx.x] = st->chg_slot[threadIdx.x]; csrc[threadIdx.x] = st->chg_src[threadIdx.x]; }
    __syncthreads();
    const int x = st->sx, xn = st->sxn, y = st->sy, yn = st->syn;
    const int xb = (xn >= 0) ? (x & ~1) : x, yb = (yn >= 0) ? (y & ~1) : y;
    Formula F{st->kind, st->fX, st->fY, st->fZ, st->fW};
    const double Duv = st->Duv;

    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < m; t += gridDim.x * blockDim.x) {
        // ---- role 1: subtract old cluster distances (old layout), bystander representatives only
        {
            const int s = t;
            const bool pPair = s < P2;
            if (!(pPair && (s & 1)) && s != xb && s != yb) {
                const double dpx = sub_dist(D, ld, s, pPair, x, xn);
                const double dpy = sub_dist(D, ld, s, pPair, y, yn);
                const double ns = (Sx[s] - dpx) - dpy;
                Sx[s] = ns;
                double nb = 0.0;
                if (pPair) { nb = (Sx[s + 1] - dpx) - dpy; Sx[s + 1] = nb; }
                for (int k = 0; k < K; ++k) {
                    if (csrc[k] == s) st->chg_Sx[k] = ns;
                    if (pPair && csrc[k] == s + 1) st->chg_Sx[k] = nb;
                }
            }
        }
        // ---- role 2: rows of the changed slots in the NEW layout, column t
        if (t < m_new) {
            int colsrc = t;
            for (int k = 0; k < K; ++k) if (cslot[k] == t) colsrc = csrc[k];
            double fu = 0.0, fv = 0.0;
            bool haveF = false;
            for (int k = 0; k < K; ++k) {
                const int rs = csrc[k];
                double v;
                if (rs >= 0) {
                    if (colsrc >= 0) v = D[(int64_t)rs * ld + colsrc];
                    else { double a, b; F.eval(D, ld, rs, a, b); v = (colsrc == SRC_NEW_U) ? a : b; }
                } else {
                    if (colsrc >= 0) {
                        if (!haveF) { F.eval(D, ld, colsrc, fu, fv); haveF = true; }
                        v = (rs == SRC_NEW_U) ? fu : fv;
                    } else v = (rs == colsrc) ? 0.0 : Duv;
                }
                scratch[(int64_t)k * ld + t] = v;
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) tl_stamp(st, TL_ROWS1);
}

// ------------------------------------------------------------------ K5b+K6a: scatter rows/cols + add sweep
// The last block to finish commits the iteration (m, c, P2, iter, done) and masks the new cluster for the next scan:
// its u.Sx is summed by k_chain + k_patch concurrently with that scan.
__global__ void __launch_bounds__(256)
k_scatter(double* D, int64_t ld, double* Sx, const int* __restrict__ pos, DevState* st, const double* __restrict__ scratch,
          double* stage, const int* __restrict__ id, const int* __restrict__ p2s) {
    if (st->done || st->skip) return;
    __shared__ bool amLast;
    if (blockIdx.x == 0 && threadIdx.x == 0) tl_stamp(st, TL_SCAT0);
    const int m_new = st->m_new, P2n = st->P2_new, K = st->K, su = st->su;
    const int Ln = (m_new + xsum::THREADS - 1) / xsum::THREADS;   // stage is segment-transposed for k_chain
    auto sidx = [&](int p) -> int { return (p % Ln) * xsum::THREADS + p / Ln; };
    __shared__ int cslot[MAXK];
    __shared__ double cSx[MAXK];
    if (threadIdx.x < MAXK) { cslot[threadIdx.x] = st->chg_slot[threadIdx.x]; cSx[threadIdx.x] = st->chg_Sx[threadIdx.x]; }
    __syncthreads();
    const double* r0 = scratch;        // row of u  (chg index 0 is always su)
    const double* r1 = scratch + ld;   // row of u' (chg index 1 is always su+1)
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < m_new; t += gridDim.x * blockDim.x) {
        for (int k = 0; k < K; ++k) {
            const double v = scratch[(int64_t)k * ld + t];
            const int s = cslot[k];
            D[(int64_t)s * ld + t] = v;
            D[(int64_t)t * ld + s] = v;
        }
        // add new cluster distances (updateClusterDistances, :517-536)
        const bool pPair = t < P2n;
        if (pPair && (t & 1)) continue;
        if (t == su) {
            stage[sidx(pos[t])] = 0.0;
            stage[sidx(pos[t + 1])] = 0.0;
            continue;
        }
        double base0 = Sx[t], base1 = pPair ? Sx[t + 1] : 0.0;
        for (int k = 0; k < K; ++k) {
            if (cslot[k] == t) base0 = cSx[k];
            if (pPair && cslot[k] == t + 1) base1 = cSx[k];
        }
        double dpu;
        if (pPair) dpu = (((r0[t] + r1[t]) + r0[t + 1]) + r1[t + 1]) * 0.25;
        else dpu = (r0[t] + r1[t]) * 0.5;
        Sx[t] = base0 + dpu;
        stage[sidx(pos[t])] = dpu;
        if (pPair) { Sx[t + 1] = base1 + dpu; stage[sidx(pos[t + 1])] = 0.0; }
    }
    // ---- commit: every block has read the event descriptor before it arrives here
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) amLast = (atomicAdd(&st->commit_ticket, 1u) == gridDim.x - 1);
    __syncthreads();
    if (amLast && threadIdx.x == 0) {
        __threadfence();
        st->commit_ticket = 0;
        tl_stamp(st, TL_SCAT1);
        st->m = m_new; st->c = st->c_new; st->P2 = P2n;
        st->iter += 1;
        st->mask_su = su;
        if (m_new <= 3) {
            st->done = 1;
            for (int i = 0; i < 3; ++i) st->final3[i] = id[p2s[i]];
        }
    }
}

// ------------------------------------------------------------------ K6b: u.Sx chain + the new cluster's pairs
// k_chain then k_patch run on a forked graph branch, concurrently with the NEXT iteration's selection scan (which reads the
// new cluster's Sx as -inf).  (1) k_chain: u.Sx = left-to-right sum of Dpu in position order (NetMakerOriginal.java:530-535),
// bit-exact; (2) k_patch: Q of (u-cluster, every other cluster) with that exact u.Sx, in the reference's role order
// (:215-226), min-loc on the same (Q, i, j) key as the scan.  k_rx_stage (after the graph join) merges the two partial min-locs.
__global__ void __launch_bounds__(PICK_THREADS, 1)
k_chain(double* Sx, DevState* st, const double* __restrict__ stage, int serial_chain, int stage_cap) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double (*buf)[1][CH_TILE] = reinterpret_cast<double (*)[1][CH_TILE]>(smem_raw);
    __shared__ double tot[1];
    if (st->done) return;
    const int tid = threadIdx.x;
    const int su = st->mask_su;
    const int m = st->m;   // committed by k_scatter
    if (tid == 0) tl_stamp(st, TL_CHAIN0);
    if (su >= 0) {
        const int Ln = (m + xsum::THREADS - 1) / xsum::THREADS;
        auto load_lin = [&](int, int i) -> double { return stage[(i % Ln) * xsum::THREADS + i / Ln]; };
        if (serial_chain) block_seq_sum<1>(buf, m, load_lin, tot);
        else if (Ln * xsum::THREADS <= stage_cap) {
            // the chain (segment-transposed, Ln x 1024) into shared memory: all of a thread's loads are independent
            double* sc = reinterpret_cast<double*>(smem_raw + CHAIN_SMEM_BASE);
            for (int k0 = 0; k0 < Ln; k0 += 8) {
                double v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) if (k0 + u < Ln) v[u] = stage[(k0 + u) * xsum::THREADS + tid];
#pragma unroll
                for (int u = 0; u < 8; ++u) if (k0 + u < Ln) sc[(k0 + u) * xsum::THREADS + tid] = v[u];
            }
            __syncthreads();
            auto load_sm = [&](int, int t, int k) -> double { return sc[k * xsum::THREADS + t]; };
            xsum::block_exact_seq_sum<1>(reinterpret_cast<xsum::SmemN<1>*>(smem_raw), m, load_sm, [](int) { return true; }, tot);
        } else {
            auto load_seg = [&](int, int t, int k) -> double { return stage[k * xsum::THREADS + t]; };
            xsum::block_exact_seq_sum<1>(reinterpret_cast<xsum::SmemN<1>*>(smem_raw), m, load_seg, [](int) { return true; }, tot);
        }
        const double Su = tot[0];
        if (tid == 0) { Sx[su] = Su; Sx[su + 1] = Su; tl_stamp(st, TL_CHAIN1); }
    }
}

// (2) of the forked branch: Q of (new cluster, every other cluster) with the exact u.Sx k_chain has just written, in the
// reference's role order, min-loc on the scan's key.  Small blocks (128 threads, no shared-memory ring) that co-reside with
// the scan's CTAs, so that all loads of the 2*m entries are in flight at once even while the scan saturates HBM; the last
// block to finish reduces the per-block partials into st->patchQ / patchKey.
constexpr int PATCH_THREADS = 128;
constexpr int PATCH_BLOCKS = 32;
__global__ void __launch_bounds__(PATCH_THREADS)
k_patch(const double* __restrict__ D, int64_t ld, const double* __restrict__ Sx, const int* __restrict__ pos, DevState* st,
        Partial* __restrict__ ppart) {
    if (st->done) return;
    __shared__ Partial wbest[PATCH_THREADS / 32];
    __shared__ bool amLast;
    const int tid = threadIdx.x;
    const int su = st->mask_su;
    const int m = st->m, P2 = st->P2;
    const bool strategy = (st->mode != 0 && m > st->fallback);
    double bq = INFINITY;
    unsigned long long bk = ~0ull;
    if (su >= 0 && !strategy && !(m == 4 && st->c == 2)) {
        const double Su = Sx[su];
        const double cm2 = (double)st->c - 2.0;
        const int posU = pos[su];
        const double* ru = D + (int64_t)su * ld;
        const double* run = ru + ld;
        constexpr int PU = 4;   // 4 independent element groups per thread: all loads of a sweep are in flight together
        const int stride = gridDim.x * PATCH_THREADS;
        for (int t0 = blockIdx.x * PATCH_THREADS + tid; t0 < m; t0 += PU * stride) {
            double a[PU], b[PU], c2[PU], d2[PU], St[PU];
            int pt[PU];
            bool use[PU], pr[PU];
#pragma unroll
            for (int u = 0; u < PU; ++u) {
                const int t = t0 + u * stride;
                pr[u] = t < P2;
                use[u] = t < m && !(pr[u] && (t & 1)) && (t & ~1) != su;   // representatives of the other clusters
                if (use[u]) {
                    pt[u] = pos[t]; St[u] = Sx[t]; a[u] = ru[t]; b[u] = run[t];
                    if (pr[u]) { c2[u] = ru[t + 1]; d2[u] = run[t + 1]; }
                }
            }
#pragma unroll
            for (int u = 0; u < PU; ++u) {
                if (!use[u]) continue;
                const bool uIsP = posU > pt[u];   // the higher position plays p (:208-213)
                double dpq;
                if (pr[u]) dpq = uIsP ? (((a[u] + c2[u]) + b[u]) + d2[u]) * 0.25 : (((a[u] + b[u]) + c2[u]) + d2[u]) * 0.25;
                else dpq = (a[u] + b[u]) * 0.5;
                const double q = uIsP ? (cm2 * dpq - Su) - St[u] : (cm2 * dpq - St[u]) - Su;
                const unsigned long long key = uIsP ? (((unsigned long long)posU << 32) | (unsigned)pt[u])
                                                    : (((unsigned long long)pt[u] << 32) | (unsigned)posU);
                if (better(q, key, bq, bk)) { bq = q; bk = key; }
            }
        }
    }
    auto warp_min = [&]() {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double oq = __shfl_down_sync(0xffffffffu, bq, off);
            const unsigned long long ok = __shfl_down_sync(0xffffffffu, bk, off);
            if (better(oq, ok, bq, bk)) { bq = oq; bk = ok; }
        }
    };
    warp_min();
    if ((tid & 31) == 0) wbest[tid >> 5] = Partial{bq, bk};
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < PATCH_THREADS / 32; ++w)
            if (better(wbest[w].q, wbest[w].key, bq, bk)) { bq = wbest[w].q; bk = wbest[w].key; }
        ppart[blockIdx.x] = Partial{bq, bk};
        __threadfence();
        amLast = (atomicAdd(&st->patch_ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (amLast && tid < 32) {
        __threadfence();
        bq = INFINITY; bk = ~0ull;
        for (int b = tid; b < (int)gridDim.x; b += 32) {
            const double pq = __ldcg(&ppart[b].q);
            const unsigned long long pk = __ldcg(&ppart[b].key);
            if (better(pq, pk, bq, bk)) { bq = pq; bk = pk; }
        }
        warp_min();
        if (tid == 0) {
            st->patchQ = bq;
            st->patchKey = bk;
            st->patch_ticket = 0;
            tl_stamp(st, TL_PATCH1);
        }
    }
}

// stand-alone entry for the exact left-to-right summation (parity tests of fnn_exact_sum.cuh)
__global__ void __launch_bounds__(PICK_THREADS, 1)
k_seqsum(const double* __restrict__ rows, int64_t stride, int nrows, int len, double* out, int serial_chain) {
    extern __shared__ unsigned char smem_raw[];
    __shared__ double res[4];
    const int L = (len + xsum::THREADS - 1) / xsum::THREADS;
    auto load = [&](int r, int i) -> double { return r < nrows ? rows[(int64_t)r * stride + i] : 0.0; };
    auto load_seg = [&](int r, int t, int k) -> double { return rows[(int64_t)r * stride + (int64_t)t * L + k]; };
    if (serial_chain) block_seq_sum<4>(reinterpret_cast<double (*)[4][CH_TILE]>(smem_raw), len, load, res);
    else xsum::block_exact_seq_sum<4>(reinterpret_cast<xsum::Smem*>(smem_raw), len, load_seg, [&](int r) { return r < nrows; }, res);
    if (threadIdx.x < nrows) out[threadIdx.x] = res[threadIdx.x];
}

}  // namespace

// ============================================================================ host side
struct fnn_ctx {
    fnn_opts o;
    int64_t n = 0, ld = 0;
    int sms = 148;
    cudaStream_t stream = nullptr;
    double* D = nullptr;
    double* Sx = nullptr;
    double* scratch = nullptr;
    double* stage = nullptr;
    double* rxs = nullptr;            // 4 staged ComputeRx rows, segment-transposed
    relaxed::Machine* rl_machine = nullptr;   // Relaxed: the control state machine and its work arrays (device)
    int *rl_rowPerm = nullptr, *rl_epoch = nullptr, *rl_clist = nullptr, *rl_loff = nullptr, *rl_lcnt = nullptr, *rl_lme = nullptr;
    int *rl_tie = nullptr, *rl_mymin = nullptr;
    int rl_max_lists = 0, rl_tie_cap = 0, rl_mymin_cap = 0;
    int* nbrpos = nullptr;            // Random modes: neighbour position per position, the walk's (i, j) pairs
    int2* pairs = nullptr;
    modes::WalkState* walk = nullptr;
    unsigned int* walk_ticket = nullptr;
    int64_t rxs_ld = 0;
    double* trace = nullptr;
    long long* record = nullptr;      // per-iteration strategy record (fnn_record.h), kept with the trace
    int *id = nullptr, *pos = nullptr, *p2s = nullptr, *amalg = nullptr;
    DevState* st = nullptr;
    Partial* partials = nullptr;      // per-block partial min-locs of k_scan_tma and k_random_eval
    int partials_cap = 0;             // ... and their number: no grid that writes them may be larger
    double* rx_part = nullptr;        // per-block partial ComputeRx sums of k_rx_stage
    Partial* patch_part = nullptr;    // per-block partial min-locs of k_patch
    int scan_grid = 0, row_grid = 0, eval_grid = 0;
    // u.Sx chain + new-cluster patch on a forked branch, concurrent with the next scan (which then leaves one SM to it)
    size_t chain_smem = 0;            // k_chain + k_patch: exact-summation workspace + (if it fits) the staged chain
    int chain_stage_cap = 0;          // elements of the chain that fit in shared memory (0: read from global)
    bool overlap = false;
    int force_exact = 0;              // A/B: always decide the pick with the exact left-to-right sums
    cudaStream_t stream2 = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    bool join_pending = false;        // a k_chain + k_patch has been issued on stream2 and not yet waited for
    int launches_per_iter() const { return 7 + (o.mode >= FNN_RANDOM_N ? 2 : 0) + (o.mode == FNN_RELAXED ? 1 : 0); }
    DevState* h_st = nullptr;  // pinned
    CUtensorMap tmap;
    bool have_tmap = false;
    int rank = 0, world = 1;
    long long run_counter = 0;
    int serial_chain = 0;             // 1: one-lane dependent chain instead of the collapsed exact summation
    Mailbox* mail = nullptr;          // this rank's mailbox (device memory, IPC-exported)
    PeerTable* peers = nullptr;       // device table of every rank's mailbox (own entry = mail)
    void* opened[MAX_WORLD] = {nullptr};
    cudaGraphExec_t graph = nullptr;
    cudaGraphExec_t graph_strategy = nullptr;   // Relaxed/Random while m > fallback: the same iterations without the (no-op) scan launch
    int graph_iters = 0;
    unsigned long long* tl = nullptr;  // debug timeline (FNN_TIMELINE)
    int tl_iter0 = 0, tl_count = 0;
    std::string tl_path;
    bool loaded = false;
    fnn_stats stats{};
    int64_t trace_rows = 0;
};

static int make_tensor_map(fnn_ctx* c);

static int ensure_device(const fnn_opts* o) {
    int cnt = 0;
    cudaError_t e = cudaGetDeviceCount(&cnt);
    if (e != cudaSuccess || cnt <= 0) {
        fnn::set_error("no CUDA device available (libfastnn has no CPU fallback): %s", cudaGetErrorString(e));
        cudaGetLastError();
        return FNN_E_NODEVICE;
    }
    int dev = o ? o->device : 0;
    if (dev < 0 || dev >= cnt) { fnn::set_error("device %d out of range (%d devices)", dev, cnt); return FNN_E_ARG; }
    FNN_CUDA(cudaSetDevice(dev));
    return FNN_OK;
}

extern "C" void fnn_default_opts(fnn_opts* o) {
    memset(o, 0, sizeof(*o));
    o->mode = FNN_CANONICAL;
    o->mult = 5;
    o->canonical_fallback = 1024;
    o->seed = 12345;
    o->use_graph = 1;
}

extern "C" const char* fnn_last_error(void) { return fnn::last_error(); }

extern "C" int fnn_device_count(void) {
    int cnt = 0;
    if (cudaGetDeviceCount(&cnt) != cudaSuccess) { cudaGetLastError(); return 0; }
    return cnt;
}

extern "C" void fnn_ctx_destroy(fnn_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->o.device);
    if (c->graph) cudaGraphExecDestroy(c->graph);
    if (c->graph_strategy) cudaGraphExecDestroy(c->graph_strategy);
    cudaFree(c->rl_machine); cudaFree(c->rl_rowPerm); cudaFree(c->rl_epoch); cudaFree(c->rl_clist); cudaFree(c->rl_loff);
    cudaFree(c->rl_lcnt); cudaFree(c->rl_lme); cudaFree(c->rl_tie); cudaFree(c->rl_mymin);
    cudaFree(c->D); cudaFree(c->Sx); cudaFree(c->scratch); cudaFree(c->stage); cudaFree(c->rxs); cudaFree(c->trace); cudaFree(c->record);
    for (int r = 0; r < MAX_WORLD; ++r) if (c->opened[r]) cudaIpcCloseMemHandle(c->opened[r]);
    cudaFree(c->mail); cudaFree(c->peers);
    cudaFree(c->nbrpos); cudaFree(c->pairs); cudaFree(c->walk); cudaFree(c->walk_ticket);
    cudaFree(c->id); cudaFree(c->pos); cudaFree(c->p2s); cudaFree(c->amalg); cudaFree(c->st); cudaFree(c->partials);
    cudaFree(c->rx_part); cudaFree(c->patch_part); cudaFree(c->tl);
    if (c->h_st) cudaFreeHost(c->h_st);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    if (c->stream2) cudaStreamDestroy(c->stream2);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

static int ctx_build(fnn_ctx* c, const fnn_opts* o, int64_t n);

extern "C" int fnn_ctx_create(const fnn_opts* o, int64_t n, fnn_ctx** out) {
    if (!out || n < 1) { fnn::set_error("fnn_ctx_create: bad arguments"); return FNN_E_ARG; }
    fnn_opts d;
    if (!o) { fnn_default_opts(&d); o = &d; }
    if (n > 2000000) { fnn::set_error("n too large"); return FNN_E_ARG; }
    if (o->mode < 0 || o->mode > FNN_RANDOM_LOGN) { fnn::set_error("unknown mode %d", o->mode); return FNN_E_ARG; }
    // a Random mode draws mult * amount pairs per iteration (NeighborNetRandom.java:31-48); with none the reference has no
    // Cx (NullPointerException) and k_random_eval would have no pair to select
    if (o->mode >= FNN_RANDOM_N && o->mult < 1) { fnn::set_error("mult %d: a Random mode needs mult >= 1", o->mult); return FNN_E_ARG; }

    int rc = ensure_device(o);
    if (rc) return rc;
    fnn_ctx* c = new fnn_ctx();
    c->o = *o;
    c->n = n;
    rc = ctx_build(c, o, n);
    if (rc) { fnn_ctx_destroy(c); return rc; }   // every failure path releases what was allocated so far
    *out = c;
    return FNN_OK;
}

static int ctx_build(fnn_ctx* c, const fnn_opts* o, int64_t n) {
    c->serial_chain = (o->reserved[1] == 1) || n > (int64_t)xsum::THREADS * xsum::LEAF_MAX;
    c->ld = (n + 15) / 16 * 16;
    cudaDeviceProp prop;
    FNN_CUDA(cudaGetDeviceProperties(&prop, o->device));
    c->sms = prop.multiProcessorCount;
#define FNN_ALLOC(ptr, bytes)                                                                  \
    do {                                                                                       \
        cudaError_t e_ = cudaMalloc((void**)&(ptr), (bytes));                                  \
        if (e_ != cudaSuccess) {                                                               \
            fnn::set_error("cudaMalloc(%zu bytes) failed: %s", (size_t)(bytes), cudaGetErrorString(e_)); \
            cudaGetLastError();                                                                \
            return FNN_E_NOMEM;                                                                \
        }                                                                                      \
    } while (0)
    FNN_ALLOC(c->D, sizeof(double) * n * c->ld);
    FNN_ALLOC(c->Sx, sizeof(double) * c->ld);
    FNN_ALLOC(c->scratch, sizeof(double) * MAXK * c->ld);
    c->rxs_ld = (int64_t)xsum::THREADS * ((n + xsum::THREADS - 1) / xsum::THREADS);
    FNN_ALLOC(c->stage, sizeof(double) * c->rxs_ld);
    FNN_ALLOC(c->rxs, sizeof(double) * 4 * c->rxs_ld);
    FNN_ALLOC(c->id, sizeof(int) * c->ld);
    FNN_ALLOC(c->pos, sizeof(int) * c->ld);
    FNN_ALLOC(c->p2s, sizeof(int) * c->ld);
    FNN_ALLOC(c->amalg, sizeof(int) * 5 * (2 * n + 8));
    FNN_ALLOC(c->st, sizeof(DevState));
    FNN_ALLOC(c->mail, sizeof(Mailbox));
    FNN_ALLOC(c->peers, sizeof(PeerTable));
    FNN_CUDA(cudaMemset(c->mail, 0, sizeof(Mailbox)));
    {
        PeerTable pt;
        memset(&pt, 0, sizeof(pt));
        pt.box[0] = c->mail;
        FNN_CUDA(cudaMemcpy(c->peers, &pt, sizeof(pt), cudaMemcpyHostToDevice));
    }
    c->overlap = (o->mode == FNN_CANONICAL) && !(o->reserved[5] & 1) && c->sms > 8;
    c->force_exact = (o->reserved[5] & 2) ? 1 : 0;
    c->scan_grid = c->sms - (c->overlap ? 1 : 0);
    c->row_grid = std::max<int>(1, std::min<int64_t>((n + 255) / 256, std::min(c->sms * 4, RX_BLOCKS_MAX)));
    c->eval_grid = c->sms * 2;
    c->partials_cap = std::max(c->scan_grid, c->eval_grid);
    FNN_ALLOC(c->partials, sizeof(Partial) * c->partials_cap);
    FNN_ALLOC(c->rx_part, sizeof(double) * 8 * RX_BLOCKS_MAX);
    FNN_ALLOC(c->patch_part, sizeof(Partial) * PATCH_BLOCKS);
    if (o->record_trace) {
        FNN_ALLOC(c->trace, sizeof(double) * 8 * (n + 8));
        FNN_ALLOC(c->record, sizeof(long long) * rec::COLS * (n + 8));
    }
    if (o->mode == FNN_RELAXED) {
        c->rl_max_lists = (int)(2 * n + 16); c->rl_tie_cap = (int)(16 * n + 65536); c->rl_mymin_cap = (int)(8 * n + 65536);
        FNN_ALLOC(c->rl_machine, sizeof(relaxed::Machine));
        FNN_ALLOC(c->rl_rowPerm, sizeof(int) * n); FNN_ALLOC(c->rl_epoch, sizeof(int) * n); FNN_ALLOC(c->rl_clist, sizeof(int) * n);
        FNN_ALLOC(c->rl_loff, sizeof(int) * c->rl_max_lists); FNN_ALLOC(c->rl_lcnt, sizeof(int) * c->rl_max_lists);
        FNN_ALLOC(c->rl_lme, sizeof(int) * c->rl_max_lists);
        FNN_ALLOC(c->rl_tie, sizeof(int) * c->rl_tie_cap); FNN_ALLOC(c->rl_mymin, sizeof(int) * 2 * c->rl_mymin_cap);
        FNN_CUDA(cudaFuncSetAttribute(modes::k_relaxed_select, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(xsum::Smem)));
    }
    if (o->mode >= FNN_RANDOM_N) {
        int lg = 0;
        for (long long p10 = 1; p10 < n; p10 *= 10) ++lg;
        const long long amount = o->mode == FNN_RANDOM_LOGN ? lg : (o->mode == FNN_RANDOM_N ? n : (long long)lg * n);
        const long long max_pairs = std::max<long long>(1, (long long)o->mult * amount) + 8;
        FNN_ALLOC(c->nbrpos, sizeof(int) * c->ld);
        FNN_ALLOC(c->pairs, sizeof(int2) * max_pairs);
        FNN_ALLOC(c->walk, sizeof(modes::WalkState));
        FNN_ALLOC(c->walk_ticket, sizeof(unsigned int));
        FNN_CUDA(cudaMemset(c->walk_ticket, 0, sizeof(unsigned int)));
    }
    if (const char* e = getenv("FNN_TIMELINE")) {   // "iter0,count,file": debugging aid, never on in production
        int i0 = 0, cnt = 0;
        char path[400];
        if (sscanf(e, "%d,%d,%399s", &i0, &cnt, path) == 3 && cnt > 0 && cnt <= 100000) {
            c->tl_iter0 = i0; c->tl_count = cnt; c->tl_path = path;
            FNN_ALLOC(c->tl, sizeof(unsigned long long) * TL_EVENTS * cnt);
            FNN_CUDA(cudaMemset(c->tl, 0, sizeof(unsigned long long) * TL_EVENTS * cnt));
        }
    }
    FNN_CUDA(cudaMallocHost((void**)&c->h_st, sizeof(DevState)));
    FNN_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    FNN_CUDA(cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking));
    FNN_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    FNN_CUDA(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
    FNN_CUDA(cudaFuncSetAttribute(k_pick, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PICK_SMEM));
    {
        const size_t want = CHAIN_SMEM_BASE + sizeof(double) * (size_t)c->rxs_ld;
        if (want <= CHAIN_SMEM_MAX) { c->chain_smem = want; c->chain_stage_cap = (int)c->rxs_ld; }
        else { c->chain_smem = CHAIN_SMEM_BASE; c->chain_stage_cap = 0; }
        FNN_CUDA(cudaFuncSetAttribute(k_chain, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CHAIN_SMEM_MAX));
    }
    int trc = make_tensor_map(c);
    if (trc) return trc;
    FNN_CUDA(cudaFuncSetAttribute(tma::k_scan_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tma::SMEM_BYTES));
    return FNN_OK;
}

static int after_load(fnn_ctx* c) {
    const int n = (int)c->n;
    k_zero_diag<<<(n + 255) / 256, 256, 0, c->stream>>>(c->D, c->ld, n);
    FNN_CUDA(cudaGetLastError());
    c->loaded = true;
    return FNN_OK;
}

extern "C" int fnn_ctx_load_host(fnn_ctx* c, const double* Dh) {
    if (!c || !Dh) { fnn::set_error("fnn_ctx_load_host: null argument"); return FNN_E_ARG; }
    FNN_CUDA(cudaSetDevice(c->o.device));
    DevEvent e0, e1;
    FNN_CUDA(e0.create()); FNN_CUDA(e1.create());
    FNN_CUDA(cudaEventRecord(e0, c->stream));
    FNN_CUDA(cudaMemcpy2DAsync(c->D, c->ld * sizeof(double), Dh, c->n * sizeof(double), c->n * sizeof(double), c->n,
                               cudaMemcpyHostToDevice, c->stream));
    FNN_CUDA(cudaEventRecord(e1, c->stream));
    int rc = after_load(c);
    FNN_CUDA(cudaStreamSynchronize(c->stream));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    c->stats.h2d_ms = ms;
    return rc;
}

// Multi-GPU upload without replicating the PCIe traffic: every rank uploads only rows [row0, row0 + nrows) of the host
// matrix; the host layer then moves the blocks between the ranks over NVLink (torch.distributed broadcast on
// fnn_ctx_matrix_ptr) and calls fnn_ctx_commit_load.
extern "C" int fnn_ctx_load_host_rows(fnn_ctx* c, const double* Dh_rows, int64_t row0, int64_t nrows) {
    if (!c || !Dh_rows || row0 < 0 || nrows < 0 || row0 + nrows > c->n) { fnn::set_error("fnn_ctx_load_host_rows: bad argument"); return FNN_E_ARG; }
    FNN_CUDA(cudaSetDevice(c->o.device));
    if (nrows > 0)
        FNN_CUDA(cudaMemcpy2DAsync(c->D + row0 * c->ld, c->ld * sizeof(double), Dh_rows, c->n * sizeof(double), c->n * sizeof(double), nrows,
                                   cudaMemcpyHostToDevice, c->stream));
    FNN_CUDA(cudaStreamSynchronize(c->stream));
    return FNN_OK;
}
extern "C" int fnn_ctx_commit_load(fnn_ctx* c) {
    if (!c) { fnn::set_error("fnn_ctx_commit_load: null argument"); return FNN_E_ARG; }
    FNN_CUDA(cudaSetDevice(c->o.device));
    int rc = after_load(c);
    FNN_CUDA(cudaStreamSynchronize(c->stream));
    return rc;
}

extern "C" int fnn_ctx_load_device(fnn_ctx* c, const double* dD, int64_t ld_src) {
    if (!c || !dD || ld_src < c->n) { fnn::set_error("fnn_ctx_load_device: bad argument"); return FNN_E_ARG; }
    FNN_CUDA(cudaSetDevice(c->o.device));
    FNN_CUDA(cudaMemcpy2DAsync(c->D, c->ld * sizeof(double), dD, ld_src * sizeof(double), c->n * sizeof(double), c->n,
                               cudaMemcpyDeviceToDevice, c->stream));
    int rc = after_load(c);
    FNN_CUDA(cudaStreamSynchronize(c->stream));
    return rc;
}

extern "C" int fnn_ctx_read_matrix(fnn_ctx* c, double* out) {
    if (!c || !out || !c->loaded) { fnn::set_error("fnn_ctx_read_matrix: no matrix loaded"); return FNN_E_STATE; }
    FNN_CUDA(cudaSetDevice(c->o.device));
    FNN_CUDA(cudaMemcpy2DAsync(out, c->n * sizeof(double), c->D, c->ld * sizeof(double), c->n * sizeof(double), c->n,
                               cudaMemcpyDeviceToHost, c->stream));
    FNN_CUDA(cudaStreamSynchronize(c->stream));
    return FNN_OK;
}

extern "C" int fnn_ctx_matrix_ptr(fnn_ctx* c, double** dptr, int64_t* ld) {
    if (!c || !dptr || !ld) { fnn::set_error("fnn_ctx_matrix_ptr: null argument"); return FNN_E_ARG; }
    *dptr = c->D; *ld = c->ld;
    return FNN_OK;
}

static_assert(PICK_THREADS == xsum::THREADS, "exact-sum block size");

// Every block of k_scan_tma and k_random_eval writes partials[blockIdx.x] and the last one reads them all: a grid larger than
// the allocation would write past its end without any fault to show it.
static inline int check_partials(fnn_ctx* c, int grid, const char* kernel) {
    if (grid <= c->partials_cap) return FNN_OK;
    fnn::set_error("%s: grid of %d blocks, but partials holds %d", kernel, grid, c->partials_cap);
    return FNN_E_STATE;
}

static inline int launch_scan(fnn_ctx* c) {
    if (int rc = check_partials(c, c->scan_grid, "k_scan_tma")) return rc;
    tma::k_scan_tma<<<c->scan_grid, tma::THREADS, tma::SMEM_BYTES, c->stream>>>(c->tmap, c->Sx, c->pos, c->st, c->partials, c->peers);
    return FNN_OK;
}

// 2-D tiled tensor map over the n x ld matrix: box = 256 columns x 8 rows, no swizzle, zero OOB fill
static int make_tensor_map(fnn_ctx* c) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    FNN_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (!fn || qres != cudaDriverEntryPointSuccess) { fnn::set_error("cuTensorMapEncodeTiled not available"); return FNN_E_CUDA; }
    cuuint64_t gdim[2] = {(cuuint64_t)c->ld, (cuuint64_t)c->n};
    cuuint64_t gstr[1] = {(cuuint64_t)c->ld * sizeof(double)};
    cuuint32_t box[2] = {(cuuint32_t)tma::BOX_W, (cuuint32_t)tma::BOX_R};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = ((EncodeFn)fn)(&c->tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, c->D, gdim, gstr, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { fnn::set_error("cuTensorMapEncodeTiled failed: %d", (int)r); return FNN_E_CUDA; }
    c->have_tmap = true;
    return FNN_OK;
}
// everything of an iteration after the scan.  The previous iteration's k_chain + k_patch (forked branch) joins here: the
// strategy kernels, the selection merge and the update all need the new cluster's exact Sx.
static inline int launch_rest(fnn_ctx* c) {
    if (c->o.mode >= FNN_RANDOM_N)
        if (int rc = check_partials(c, c->eval_grid, "k_random_eval")) return rc;
    if (c->join_pending) { cudaStreamWaitEvent(c->stream, c->ev_join, 0); c->join_pending = false; }
    if (c->o.mode >= FNN_RANDOM_N) {
        modes::k_random_walk<<<1, modes::THREADS, 0, c->stream>>>(c->pos, c->p2s, c->st, c->nbrpos, c->pairs, c->walk, c->record);
        modes::k_random_eval<<<c->eval_grid, 256, 0, c->stream>>>(c->D, c->ld, c->Sx, c->p2s, c->st, c->pairs, c->walk, c->partials,
                                                                  c->walk_ticket, c->record);
    }
    if (c->o.mode == FNN_RELAXED)
        modes::k_relaxed_select<<<1, modes::THREADS, sizeof(xsum::Smem), c->stream>>>(c->D, c->ld, c->Sx, c->id, c->pos, c->p2s, c->st,
                                                                                     c->rl_machine, (int)c->n, c->record);
    k_rx_stage<<<c->row_grid, 256, 0, c->stream>>>(c->D, c->ld, c->id, c->pos, c->p2s, c->st, c->mail, c->rxs, c->rxs_ld, c->rx_part);
    k_pick<<<1, PICK_THREADS, PICK_SMEM, c->stream>>>(c->D, c->ld, c->Sx, c->id, c->pos, c->p2s, c->st, c->amalg, c->trace,
                                                    c->serial_chain, c->rxs, c->rxs_ld, c->rx_part, c->row_grid, c->force_exact);
    k_rows<<<c->row_grid, 256, 0, c->stream>>>(c->D, c->ld, c->Sx, c->st, c->scratch);
    k_scatter<<<c->row_grid, 256, 0, c->stream>>>(c->D, c->ld, c->Sx, c->pos, c->st, c->scratch, c->stage, c->id, c->p2s);
    cudaStream_t cs = c->stream;
    if (c->overlap) {
        cudaEventRecord(c->ev_fork, c->stream);
        cudaStreamWaitEvent(c->stream2, c->ev_fork, 0);
        cs = c->stream2;
    }
    k_chain<<<1, PICK_THREADS, c->chain_smem, cs>>>(c->Sx, c->st, c->stage, c->serial_chain, c->chain_stage_cap);
    k_patch<<<PATCH_BLOCKS, PATCH_THREADS, 0, cs>>>(c->D, c->ld, c->Sx, c->pos, c->st, c->patch_part);
    if (c->overlap) { cudaEventRecord(c->ev_join, c->stream2); c->join_pending = true; }
    return FNN_OK;
}
// the forked branch has to be back on the main stream before a capture ends, before the state is read, before the next run
static inline void join_branch(fnn_ctx* c) {
    if (c->join_pending) { cudaStreamWaitEvent(c->stream, c->ev_join, 0); c->join_pending = false; }
}

// expandNodes (NetMakerOriginal.java:246-325) on the host from the amalgamation log
static bool expand_order(int64_t n, const std::vector<int>& lg, int n_amalg, const int* final3, int32_t* ordering) {
    const int maxid = (int)n + 2 * n_amalg + 2;
    std::vector<int> ch1(maxid + 1, 0), ch2(maxid + 1, 0), nbr(maxid + 1, 0), nxt(maxid + 1, 0), prv(maxid + 1, 0);
    for (int k = 0; k < n_amalg; ++k) {
        const int* e = &lg[5 * k];
        ch1[e[0]] = e[2]; ch2[e[0]] = e[3];
        ch1[e[1]] = e[3]; ch2[e[1]] = e[4];
        nbr[e[0]] = e[1]; nbr[e[1]] = e[0];
    }
    int x = final3[0], y = final3[1], z = final3[2];
    nxt[x] = y; nxt[y] = z; nxt[z] = x;
    prv[x] = z; prv[y] = x; prv[z] = y;
    for (int k = n_amalg - 1; k >= 0; --k) {
        int u = lg[5 * k], v = nbr[u];
        x = ch1[u]; y = ch2[u]; z = ch2[v];
        if (v != nxt[u]) { std::swap(u, v); std::swap(x, z); }
        prv[x] = prv[u]; nxt[prv[x]] = x;
        nxt[x] = y; prv[y] = x;
        nxt[y] = z; prv[z] = y;
        nxt[z] = nxt[v]; prv[nxt[z]] = z;
    }
    for (int64_t guard = 0; x != 1; ++guard) {   // rotate to taxon 1 (:312-316); a damaged log must not spin forever
        if (guard > n) return false;
        x = nxt[x];
    }
    int a = x, t = 0;
    ordering[0] = 0;
    do { ordering[++t] = a; a = nxt[a]; } while (a != x && t < n);
    return a == x && t == n;
}

extern "C" int fnn_ctx_order(fnn_ctx* c, int32_t* ordering) {
    if (!c || !ordering) { fnn::set_error("fnn_ctx_order: null argument"); return FNN_E_ARG; }
    const int64_t n = c->n;
    if (n <= 3) {  // NetMakerOriginal.java:133-140
        for (int64_t i = 0; i <= n; ++i) ordering[i] = (int32_t)i;
        return FNN_OK;
    }
    if (!c->loaded) { fnn::set_error("fnn_ctx_order: no matrix loaded"); return FNN_E_STATE; }
    FNN_CUDA(cudaSetDevice(c->o.device));
    c->loaded = false;  // the matrix is consumed
    DevEvent e0, e1;
    FNN_CUDA(e0.create()); FNN_CUDA(e1.create());
    FNN_CUDA(cudaEventRecord(e0, c->stream));
    const int ni = (int)n;
    k_init_nodes<<<(ni + 255) / 256, 256, 0, c->stream>>>(ni, c->id, c->pos, c->p2s, c->st, c->o.mode, c->o.mult,
                                                          c->o.canonical_fallback, (long long)c->o.seed, c->rank, c->world, (long long)(++c->run_counter) << 32,
                                                          c->tl, c->tl_iter0, c->tl_count);
    k_rowsum<<<(ni + 127) / 128, 128, 0, c->stream>>>(c->D, c->ld, ni, c->Sx, c->st);
    FNN_CUDA(cudaGetLastError());
    // iterations in which no strategy runs keep a zero record row; the strategy kernels fill the others
    if (c->record) FNN_CUDA(cudaMemsetAsync(c->record, 0, sizeof(long long) * rec::COLS * (n + 8), c->stream));
    int64_t launches = 2, scans = 0;
    const int64_t max_iters = n;  // n-3 .. n-1 iterations; kernels no-op once done
    double prof_ms = 0.0, prof_bytes = 0.0;
    int64_t prof_samples = 0;

    if (c->o.mode == FNN_RELAXED) {   // (re)initialise the device-side control state machine (NeighborNetLocal.java:26-32)
        relaxed::Machine M;
        memset(&M, 0, sizeof(M));
        M.rng = ((unsigned long long)c->o.seed ^ 0x5DEECE66DULL) & ((1ULL << 48) - 1);   // java.util.Random(seed)
        M.first_time = 1;
        M.rowPerm = c->rl_rowPerm; M.cache_epoch = c->rl_epoch; M.cache_list = c->rl_clist;
        M.list_off = c->rl_loff; M.list_cnt = c->rl_lcnt; M.list_me = c->rl_lme; M.tiepool = c->rl_tie; M.mymin = c->rl_mymin;
        M.max_lists = c->rl_max_lists; M.tie_cap = c->rl_tie_cap; M.mymin_cap = c->rl_mymin_cap;
        M.additive = c->o.additive ? 1 : 0;
        M.cx_pos = M.cy_pos = -1;
        FNN_CUDA(cudaMemsetAsync(c->rl_epoch, 0, sizeof(int) * n, c->stream));
        FNN_CUDA(cudaMemcpyAsync(c->rl_machine, &M, sizeof(M), cudaMemcpyHostToDevice, c->stream));
        FNN_CUDA(cudaStreamSynchronize(c->stream));
    }
    if (c->o.profile_every > 0) {
        // sampled per-launch timing of the selection kernel (roofline.achieved in bench.py)
        DevEvent p0, p1;
        FNN_CUDA(p0.create()); FNN_CUDA(p1.create());
        for (int64_t it = 0; it < max_iters; ++it) {
            const bool sample = (it % c->o.profile_every) == 0;
            if (sample) {
                join_branch(c);
                FNN_CUDA(cudaMemcpyAsync(c->h_st, c->st, sizeof(DevState), cudaMemcpyDeviceToHost, c->stream));
                FNN_CUDA(cudaStreamSynchronize(c->stream));
                if (c->h_st->done) break;
                FNN_CUDA(cudaEventRecord(p0, c->stream));
            }
            if (int rc = launch_scan(c)) return rc;
            if (sample) {
                FNN_CUDA(cudaEventRecord(p1, c->stream));
                FNN_CUDA(cudaEventSynchronize(p1));
                float ms = 0;
                cudaEventElapsedTime(&ms, p0, p1);
                const double mm = c->h_st->m, pp = c->h_st->P2 / 2;
                prof_ms += ms;
                prof_bytes += 4.0 * mm * (mm - 1.0) - 8.0 * pp + 8.0 * mm;
                ++prof_samples;
            }
            if (int rc = launch_rest(c)) return rc;
            launches += c->launches_per_iter(); ++scans;
        }
        join_branch(c);
        FNN_CUDA(cudaGetLastError());
    } else if (c->o.use_graph) {
        constexpr int GI = 32;  // iterations per graph
        if (!c->graph) {
            cudaGraph_t g;
            int rc = FNN_OK;
            FNN_CUDA(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
            for (int i = 0; i < GI && !rc; ++i) { rc = launch_scan(c); if (!rc) rc = launch_rest(c); }
            join_branch(c);
            FNN_CUDA(cudaStreamEndCapture(c->stream, &g));
            if (rc) { cudaGraphDestroy(g); return rc; }
            FNN_CUDA(cudaGraphInstantiate(&c->graph, g, 0));
            cudaGraphDestroy(g);
            c->graph_iters = GI;
            if (c->o.mode != FNN_CANONICAL) {
                FNN_CUDA(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
                for (int i = 0; i < GI && !rc; ++i) rc = launch_rest(c);
                join_branch(c);
                FNN_CUDA(cudaStreamEndCapture(c->stream, &g));
                if (rc) { cudaGraphDestroy(g); return rc; }
                FNN_CUDA(cudaGraphInstantiate(&c->graph_strategy, g, 0));
                cudaGraphDestroy(g);
            }
        }
        int64_t it = 0;
        int64_t m_known = n;   // active nodes at the last poll; an iteration removes at most 2
        while (it < max_iters) {
            // graphs between done-flag polls.  While every iteration of the batch is certain to run the strategy
            // (m > fallback throughout), the graph without the no-op canonical scan launch is replayed.
            const int64_t batch = c->graph_strategy ? 16 : 64;
            const bool strategy_only = c->graph_strategy && (m_known - 2 * batch * GI > (int64_t)c->o.canonical_fallback);
            for (int64_t b = 0; b < batch && it < max_iters; ++b, it += GI) {
                FNN_CUDA(cudaGraphLaunch(strategy_only ? c->graph_strategy : c->graph, c->stream));
                launches += (int64_t)(c->launches_per_iter() - (strategy_only ? 1 : 0)) * GI;
                if (!strategy_only) scans += GI;
            }
            FNN_CUDA(cudaMemcpyAsync(c->h_st, c->st, sizeof(DevState), cudaMemcpyDeviceToHost, c->stream));
            FNN_CUDA(cudaStreamSynchronize(c->stream));
            if (c->h_st->done) break;
            m_known = c->h_st->m;
        }
    } else {
        int64_t it = 0;
        while (it < max_iters) {
            for (int b = 0; b < 256 && it < max_iters; ++b, ++it) {
                if (int rc = launch_scan(c)) return rc;
                if (int rc = launch_rest(c)) return rc;
                launches += c->launches_per_iter(); ++scans;
            }
            join_branch(c);
            FNN_CUDA(cudaGetLastError());
            FNN_CUDA(cudaMemcpyAsync(c->h_st, c->st, sizeof(DevState), cudaMemcpyDeviceToHost, c->stream));
            FNN_CUDA(cudaStreamSynchronize(c->stream));
            if (c->h_st->done) break;
        }
    }
    join_branch(c);
    FNN_CUDA(cudaMemcpyAsync(c->h_st, c->st, sizeof(DevState), cudaMemcpyDeviceToHost, c->stream));
    FNN_CUDA(cudaEventRecord(e1, c->stream));
    FNN_CUDA(cudaStreamSynchronize(c->stream));
    FNN_CUDA(cudaStreamSynchronize(c->stream2));
    FNN_CUDA(cudaGetLastError());
    if (c->h_st->error) {
        fnn::set_error("device-side failure, code %d (10 = no pair found, 11/13 = tie or list pool overflow, 12 = candidate pool overflow, "
                       "21 = certified pick disagrees with the exact sums, 30 = a peer rank never posted its partial min-loc)", c->h_st->error);
        return FNN_E_STATE;
    }
    if (!c->h_st->done) { fnn::set_error("agglomeration did not terminate (m=%d after %d iterations)", c->h_st->m, c->h_st->iter); return FNN_E_STATE; }
    if (c->tl) {   // dump the timeline window (ns since its first stamp)
        std::vector<unsigned long long> h((size_t)TL_EVENTS * c->tl_count);
        FNN_CUDA(cudaMemcpy(h.data(), c->tl, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        const std::string path = c->world > 1 ? c->tl_path + ".r" + std::to_string(c->rank) : c->tl_path;
        if (FILE* f = fopen(path.c_str(), "w")) {
            fprintf(f, "iter,scan0,scan1,rx0,rx1,pick0,pick1,rows0,rows1,scat0,scat1,chain0,chain1,patch1,sel0,sel1\n");
            unsigned long long base = 0;
            for (size_t i = 0; i < h.size() && !base; ++i) base = h[i];
            for (int k = 0; k < c->tl_count; ++k) {
                fprintf(f, "%d", c->tl_iter0 + k);
                for (int e = 0; e < 15; ++e) {
                    const unsigned long long v = h[(size_t)k * TL_EVENTS + e];
                    fprintf(f, ",%lld", v ? (long long)(v - base) : -1ll);
                }
                fprintf(f, "\n");
            }
            fclose(f);
        }
    }
    const int n_amalg = c->h_st->n_amalg;
    std::vector<int> lg(5 * (size_t)std::max(n_amalg, 1));
    FNN_CUDA(cudaMemcpy(lg.data(), c->amalg, sizeof(int) * 5 * n_amalg, cudaMemcpyDeviceToHost));
    if (!expand_order(n, lg, n_amalg, c->h_st->final3, ordering)) {
        fnn::set_error("amalgamation log does not expand to a cycle over %lld taxa", (long long)n);
        return FNN_E_STATE;
    }
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    c->stats.order_ms = ms;
    c->stats.iterations = c->h_st->iter;
    c->stats.kernel_launches = launches;
    c->stats.scan_launches = scans;
    c->stats.scan_alg_bytes = c->h_st->alg_bytes;
    c->stats.prof_scan_ms = prof_ms;
    c->stats.prof_scan_bytes = prof_bytes;
    c->stats.prof_scan_samples = prof_samples;
    c->stats.reserved[0] = (double)c->h_st->cert_ok;     // picks decided by the bounded parallel ComputeRx sums
    c->stats.reserved[1] = (double)c->h_st->cert_fail;   // picks that needed the exact left-to-right sums
    c->stats.reserved[2] = (double)c->h_st->strat_bytes; // Relaxed row scans / Random samples: algorithmic bytes (SURVEY 8d K7/K9)
    c->stats.reserved[3] = (double)c->h_st->strat_units; // ... and their number
    c->trace_rows = c->h_st->iter;
    return FNN_OK;
}

extern "C" int64_t fnn_ctx_trace(fnn_ctx* c, double* rows, int64_t max_rows) {
    if (!c || !rows || !c->trace) { fnn::set_error("fnn_ctx_trace: trace not recorded (opts.record_trace)"); return FNN_E_STATE; }
    cudaSetDevice(c->o.device);
    int64_t k = std::min<int64_t>(c->trace_rows, max_rows);
    if (cudaMemcpy(rows, c->trace, sizeof(double) * 8 * k, cudaMemcpyDeviceToHost) != cudaSuccess) {
        fnn::set_error("trace copy failed: %s", cudaGetErrorString(cudaGetLastError()));
        return FNN_E_CUDA;
    }
    return k;
}

extern "C" int64_t fnn_ctx_strategy_record(fnn_ctx* c, int64_t* rows, int64_t max_rows) {
    if (!c || !rows || !c->record) { fnn::set_error("fnn_ctx_strategy_record: record not kept (opts.record_trace)"); return FNN_E_STATE; }
    cudaSetDevice(c->o.device);
    int64_t k = std::min<int64_t>(c->trace_rows, max_rows);
    if (cudaMemcpy(rows, c->record, sizeof(long long) * rec::COLS * k, cudaMemcpyDeviceToHost) != cudaSuccess) {
        fnn::set_error("strategy record copy failed: %s", cudaGetErrorString(cudaGetLastError()));
        return FNN_E_CUDA;
    }
    return k;
}

extern "C" int fnn_ctx_stats(fnn_ctx* c, fnn_stats* out) {
    if (!c || !out) { fnn::set_error("fnn_ctx_stats: null argument"); return FNN_E_ARG; }
    *out = c->stats;
    return FNN_OK;
}

extern "C" int fnn_rowsums(const fnn_opts* o, const double* Dh, int64_t n, double* Sx_out) {
    fnn_ctx* c = nullptr;
    int rc = fnn_ctx_create(o, n, &c);
    if (rc) return rc;
    rc = fnn_ctx_load_host(c, Dh);
    if (!rc) {
        k_rowsum<<<((int)n + 127) / 128, 128, 0, c->stream>>>(c->D, c->ld, (int)n, c->Sx, nullptr);
        if (cudaMemcpyAsync(Sx_out, c->Sx, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
            cudaStreamSynchronize(c->stream) != cudaSuccess) {
            fnn::set_error("fnn_rowsums: %s", cudaGetErrorString(cudaGetLastError()));
            rc = FNN_E_CUDA;
        }
    }
    fnn_ctx_destroy(c);
    return rc;
}

// internal accessors for the other translation units of the library (not part of the ABI)
int64_t fnn_ctx_n_(fnn_ctx* c) { return c->n; }
void fnn_ctx_mark_loaded_(fnn_ctx* c) { c->loaded = true; }
int fnn_ctx_device_(fnn_ctx* c) { return c->o.device; }
int fnn_ctx_sms_(fnn_ctx* c) { return c->sms; }
cudaStream_t fnn_ctx_stream_(fnn_ctx* c) { return c->stream; }

extern "C" int fnn_seq_sum(const fnn_opts* o, const double* rows, int32_t nrows, int64_t len, double* out) {
    if (!rows || !out || nrows < 1 || nrows > 4 || len < 0 || len > (int64_t)xsum::THREADS * xsum::LEAF_MAX) { fnn::set_error("fnn_seq_sum: bad arguments"); return FNN_E_ARG; }
    int rc = ensure_device(o);
    if (rc) return rc;
    double *d_rows = nullptr, *d_out = nullptr;
    DevScratch scratch;   // freed on every exit path
    FNN_CUDA(scratch.alloc((void**)&d_rows, sizeof(double) * (size_t)nrows * (size_t)std::max<int64_t>(len, 1)));
    FNN_CUDA(scratch.alloc((void**)&d_out, sizeof(double) * 4));
    FNN_CUDA(cudaMemcpy(d_rows, rows, sizeof(double) * (size_t)nrows * (size_t)len, cudaMemcpyHostToDevice));
    FNN_CUDA(cudaFuncSetAttribute(k_seqsum, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PICK_SMEM));
    k_seqsum<<<1, PICK_THREADS, PICK_SMEM>>>(d_rows, len, nrows, (int)len, d_out, o ? o->reserved[1] : 0);
    FNN_CUDA(cudaGetLastError());
    if (o && o->reserved[2] > 0 && getenv("FNN_DEBUG")) {   // kernel-only timing for profiling sessions
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0); cudaEventCreate(&e1);
        cudaEventRecord(e0);
        for (int i = 0; i < o->reserved[2]; ++i)
            k_seqsum<<<1, PICK_THREADS, PICK_SMEM>>>(d_rows, len, nrows, (int)len, d_out, o->reserved[1]);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        fprintf(stderr, "[fnn] k_seqsum nrows=%d len=%lld serial=%d: %.2f us/launch\n", nrows, (long long)len, o->reserved[1],
                1e3 * ms / o->reserved[2]);
        cudaEventDestroy(e0); cudaEventDestroy(e1);
    }
    FNN_CUDA(cudaMemcpy(out, d_out, sizeof(double) * nrows, cudaMemcpyDeviceToHost));
    return FNN_OK;
}

// ---- multi-GPU wiring: one process per GPU; the host language layer moves the 64-byte IPC handles
extern "C" int fnn_ctx_ipc_handle(fnn_ctx* c, void* handle_out) {
    if (!c || !handle_out) { fnn::set_error("fnn_ctx_ipc_handle: null argument"); return FNN_E_ARG; }
    FNN_CUDA(cudaSetDevice(c->o.device));
    cudaIpcMemHandle_t h;
    FNN_CUDA(cudaIpcGetMemHandle(&h, c->mail));
    memcpy(handle_out, &h, sizeof(h));
    return FNN_OK;
}

extern "C" int fnn_ctx_connect(fnn_ctx* c, int32_t rank, int32_t world, const void* handles) {
    if (!c || !handles || world < 1 || world > MAX_WORLD || rank < 0 || rank >= world) {
        fnn::set_error("fnn_ctx_connect: need 0 <= rank < world <= %d", MAX_WORLD);
        return FNN_E_ARG;
    }
    FNN_CUDA(cudaSetDevice(c->o.device));
    for (int r = 0; r < MAX_WORLD; ++r)   // a second connect replaces the first wiring
        if (c->opened[r]) { cudaIpcCloseMemHandle(c->opened[r]); c->opened[r] = nullptr; }
    PeerTable pt;
    memset(&pt, 0, sizeof(pt));
    for (int r = 0; r < world; ++r) {
        if (r == rank) { pt.box[r] = c->mail; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char*)handles + (size_t)r * sizeof(h), sizeof(h));
        void* p = nullptr;
        FNN_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        c->opened[r] = p;
        pt.box[r] = (Mailbox*)p;
    }
    FNN_CUDA(cudaMemcpy(c->peers, &pt, sizeof(pt), cudaMemcpyHostToDevice));
    c->rank = rank;
    c->world = world;
    if (c->graph) { cudaGraphExecDestroy(c->graph); c->graph = nullptr; }
    if (c->graph_strategy) { cudaGraphExecDestroy(c->graph_strategy); c->graph_strategy = nullptr; }
    return FNN_OK;
}
