// ============================================================================
// oracle/nnet_oracle.cpp — CPU restatement of the FastNeighborNet hot path.
//
// TEST INFRASTRUCTURE ONLY.  Nothing in the product path (fastneighbornet_b200/,
// csrc/, include/) may import, link or execute this file.  Only tests/,
// __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg
// use it, and only as the checker / the timed CPU baseline.
//
// PARITY UNPINNED: the reference (pure Java 7, no tests, no fixtures, no golden
// vectors; no JVM in this image) cannot be executed here and ships nothing to
// pin against.  Fidelity rests on (i) line-by-line correspondence with the
// cited Java, (ii) an independently written object-style Python transliteration
// (oracle/pyref.py) that must agree bit-for-bit, (iii) restatement-independent
// invariants (tests/test_oracle_invariants.py) and scipy NNLS for the weights.
//
// Arithmetic contract: IEEE-754 binary64, no FMA contraction (build with
// -ffp-contract=off), sums in the reference's sequential order.
//
// Citations are file:line into /root/reference (read-only, not shipped).
// ============================================================================
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <vector>

// the PRODUCT's resumable state machine for the Relaxed control flow, compiled here for the CPU so that it can be
// held against the literal findNodes below (tests/test_relaxed_sm_cpu.py); the oracle never depends on it otherwise
#include "../fastneighbornet_b200/csrc/fnn_relaxed_sm.h"
#include "../fastneighbornet_b200/csrc/fnn_tile_iter.h"
// the digest of the product's per-iteration strategy record (fnn_ctx_strategy_record)
#include "../fastneighbornet_b200/csrc/fnn_record.h"

namespace {
static int g_use_relaxed_sm = 0;

// ---- java.util.Random (documented LCG) -------------------------------------
// RNG contract for Relaxed/Random: the reference uses the unseedable
// ThreadLocalRandom (NeighborNetLocal.java:30, NeighborNetRandom.java:27); the
// field is typed java.util.Random and the commented line :28 shows the seeded
// form.  We consume java.util.Random(seed) in exactly the reference call order.
struct JavaRandom {
    uint64_t s;
    explicit JavaRandom(int64_t seed) { s = ((uint64_t)seed ^ 0x5DEECE66DULL) & ((1ULL << 48) - 1); }
    int32_t next(int bits) {
        s = (s * 0x5DEECE66DULL + 0xBULL) & ((1ULL << 48) - 1);
        return (int32_t)((int64_t)s >> (48 - bits));
    }
    int32_t nextInt(int32_t bound) {
        int32_t r = next(31);
        int32_t m = bound - 1;
        if ((bound & m) == 0) {
            r = (int32_t)(((int64_t)bound * (int64_t)r) >> 31);
        } else {
            for (int32_t u = r;; u = next(31)) {
                r = u % bound;
                // Java int arithmetic wraps; do it in uint32 then reinterpret.
                int32_t t = (int32_t)((uint32_t)u - (uint32_t)r + (uint32_t)m);
                if (t >= 0) break;
            }
        }
        return r;
    }
};

// ---- NetNode (NetNode.java:5-15) as a struct-of-handles --------------------
struct Node {
    int id = 0;
    int64_t dist = 0;   // distID: row of D
    int pos = -1;       // positionID: slot in the active list
    int nbr = -1, ch1 = -1, ch2 = -1, next = -1, prev = -1;
    double Sx = 0.0;
};

enum Mode { CANONICAL = 0, RELAXED = 1, RANDOM_N = 2, RANDOM_NLOGN = 3, RANDOM_LOGN = 4 };

struct TraceRow {          // one per agglomeration iteration
    int32_t m, c, cx_id, cy_id, x_id, y_id, kind;   // kind: 2,3,4 ; 5 = special 4/2 case
    double best;
};

struct RowMin { int me, row; double value; };

// A fixed pool like the reference's Executors.newFixedThreadPool (FastNN.java:291-295): workers persist across
// iterations, so the timed CPU baseline pays a wake-up per slice, not a thread creation.
struct SlicePool {
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_go, cv_done;
    std::function<void(int)> job;
    int generation = 0, pending = 0;
    bool stop = false;
    explicit SlicePool(int T) {
        for (int t = 1; t < T; ++t)
            workers.emplace_back([this, t] {
                int seen = 0;
                while (true) {
                    std::function<void(int)> f;
                    {
                        std::unique_lock<std::mutex> lk(mu);
                        cv_go.wait(lk, [&] { return stop || generation != seen; });
                        if (stop) return;
                        seen = generation;
                        f = job;
                    }
                    f(t);
                    {
                        std::lock_guard<std::mutex> lk(mu);
                        if (--pending == 0) cv_done.notify_one();
                    }
                }
            });
    }
    void run(const std::function<void(int)>& f) {   // slices 1..T-1 on the workers, slice 0 here
        {
            std::lock_guard<std::mutex> lk(mu);
            job = f;
            pending = (int)workers.size();
            ++generation;
        }
        cv_go.notify_all();
        f(0);
        std::unique_lock<std::mutex> lk(mu);
        cv_done.wait(lk, [&] { return pending == 0; });
    }
    ~SlicePool() {
        { std::lock_guard<std::mutex> lk(mu); stop = true; }
        cv_go.notify_all();
        for (auto& w : workers) w.join();
    }
};

struct Engine {
    int64_t n;
    double* D;             // n*n row-major, mutated in place like the Java double[][]
    std::vector<Node> nd;  // all nodes ever created (handles are indices)
    std::vector<int> act;  // netNodes[]: handle per position, -1 = null
    std::vector<int> stack;  // amalgs
    int Cx = -1, Cy = -1;
    double best = 0.0;
    int mode = CANONICAL;
    int mult = 5;
    bool additive = false;
    int fallback = 1024;
    JavaRandom rng{0};
    // relaxed state (NeighborNetLocal.java:17-19)
    std::vector<int> rowPerm;
    bool firstTime = true;
    int top = 0;
    int64_t npe_would_fire = 0;   // times the shipped -additive loop would have NPE'd (F7)
    int64_t pair_evals = 0;
    double alg_bytes = 0.0;      // sum over canonical scans of 8 B per cross-cluster entry (SURVEY §8d)
    int threads = 1;             // >1: NeighborNetCanonical's thread-pool partition (NeighborNetCanonical.java:180-206)
    std::unique_ptr<SlicePool> pool;
    std::vector<TraceRow>* trace = nullptr;
    std::vector<int64_t>* record = nullptr;   // rec::COLS per iteration, as fnn_ctx_strategy_record returns it
    int64_t* rec_row = nullptr;               // this iteration's row (null: no record kept)
    int status = 0;
    int64_t max_iters = 0;       // >0: stop after this many agglomeration iterations (the ordering is then undefined)
    bool stopped = false;

    inline double& d(int a, int b) { return D[nd[a].dist * n + nd[b].dist]; }

    // the 1/2/4-term cluster distance, role order p then q
    // (NetMakerOriginal.java:218-225 and every copy of that ladder)
    inline double clusterDist(int p, int q) {
        const Node& P = nd[p];
        const Node& Q = nd[q];
        if (P.nbr < 0 && Q.nbr < 0) return d(p, q);
        if (P.nbr >= 0 && Q.nbr < 0) return (d(p, q) + d(P.nbr, q)) / 2.0;
        if (P.nbr < 0 && Q.nbr >= 0) return (d(p, q) + d(p, Q.nbr)) / 2.0;
        return (d(p, q) + d(p, Q.nbr) + d(P.nbr, q) + d(P.nbr, Q.nbr)) / 4.0;
    }
    inline bool isRep(int p) { return nd[p].nbr < 0 || nd[nd[p].nbr].id > nd[p].id; }

    // NetMakerOriginal.java:164-191
    void initialize(int num_nodes) {
        for (int pi = 0; pi < (int)act.size(); ++pi) {
            int p = act[pi];
            if (nd[p].nbr < 0 || nd[nd[p].nbr].id > nd[p].id) {
                for (int j = nd[p].pos + 1; j < num_nodes; ++j) {
                    int q = act[j];
                    if (nd[q].nbr < 0 || ((nd[nd[q].nbr].id > nd[q].id) && (nd[q].nbr != p))) {
                        double Dpq = clusterDist(p, q);
                        nd[p].Sx += Dpq;
                        if (nd[p].nbr >= 0) nd[nd[p].nbr].Sx += Dpq;
                        nd[q].Sx += Dpq;
                        if (nd[q].nbr >= 0) nd[nd[q].nbr].Sx += Dpq;
                    }
                }
            }
        }
    }

    // NetMakerOriginal.java:197-236 == NeighborNetCanonical.java:150-179
    void findNodesDefault(int num_active, int num_clusters) {
        Cx = Cy = -1;
        best = 1.7976931348623157e308;
        for (int i = 0; i < num_active; ++i) {
            int p = act[i];
            if (nd[p].nbr >= 0 && nd[nd[p].nbr].id < nd[p].id) continue;
            for (int j = 0; j != i; ++j) {
                int q = act[j];
                if (nd[q].nbr >= 0 && nd[nd[q].nbr].id < nd[q].id) continue;
                if (nd[q].nbr == p) continue;
                double Dpq = clusterDist(p, q);
                double Qpq = ((double)num_clusters - 2.0) * Dpq - nd[p].Sx - nd[q].Sx;
                ++pair_evals;
                if ((Cx < 0 || (Qpq < best)) && (nd[p].nbr != q)) {
                    Cx = p; Cy = q; best = Qpq;
                }
            }
        }
    }

    // NeighborNetCanonical.java:180-206 + FindNodesMulti (:50-132): the 1-based triangular pair
    // index [1, m(m-1)/2] is cut into `threads` equal slices.  The reference merges the slices
    // through a synchronized strict `<` in thread-completion order (nondeterministic on exact
    // ties, SURVEY F9); here slices are merged in slice order with strict `<`, which is the
    // 1-thread result.  Used only for the timed CPU baseline.
    void findNodesCanonicalMT(int num_active, int num_clusters) {
        Cx = Cy = -1;
        best = 1.7976931348623157e308;
        const int T = threads;
        std::vector<int> bx(T, -1), by(T, -1);
        std::vector<double> bb(T, 1.7976931348623157e308);
        const int64_t work = (int64_t)num_active * (num_active - 1) / 2;
        auto slice = [&](int t) {
            // slice [lo, hi) of the 0-based linear index over (i, j<i), i-major
            const int64_t lo = work * t / T, hi = work * (t + 1) / T;
            int i = (int)((1.0 + std::sqrt(1.0 + 8.0 * (double)lo)) / 2.0);
            while ((int64_t)i * (i - 1) / 2 > lo) --i;
            while ((int64_t)(i + 1) * i / 2 <= lo) ++i;
            int j = (int)(lo - (int64_t)i * (i - 1) / 2);
            int lx = -1, ly = -1; double lb = 1.7976931348623157e308;
            for (int64_t k = lo; k < hi; ++k) {
                int p = act[i], q = act[j];
                if (!(nd[p].nbr >= 0 && nd[nd[p].nbr].id < nd[p].id) &&
                    !(nd[q].nbr >= 0 && nd[nd[q].nbr].id < nd[q].id) && nd[q].nbr != p) {
                    double Dpq = clusterDist(p, q);
                    double Qpq = ((double)num_clusters - 2.0) * Dpq - nd[p].Sx - nd[q].Sx;
                    if (lx < 0 || Qpq < lb) { lx = p; ly = q; lb = Qpq; }
                }
                if (++j == i) { ++i; j = 0; }
            }
            bx[t] = lx; by[t] = ly; bb[t] = lb;
        };
        if (!pool) pool.reset(new SlicePool(T));
        pool->run(slice);
        for (int t = 0; t < T; ++t)
            if (bx[t] >= 0 && (Cx < 0 || bb[t] < best)) { Cx = bx[t]; Cy = by[t]; best = bb[t]; }
    }

    // ---- Relaxed (NeighborNetLocal.java) -----------------------------------
    typedef std::unordered_map<int, int> RowCache;     // node handle -> list index
    std::vector<std::vector<RowMin>> lists;

    // NeighborNetLocal.java:88-157, single-thread branch (:97-126)
    int findRowMin(int p, RowCache& found, int num_active, int num_clusters) {
        auto it = found.find(p);
        if (it != found.end()) return it->second;
        if (nd[p].nbr >= 0) {
            auto it2 = found.find(nd[p].nbr);
            if (it2 != found.end()) return it2->second;
        }
        std::vector<RowMin> mins;
        double myMin = 1.7976931348623157e308;
        for (int row = 0; row < num_active; ++row) {
            int q = act[row];
            if (p == q || (nd[p].nbr >= 0 && nd[p].nbr == q)) continue;
            double Dpq = clusterDist(p, q);
            double Qpq = ((double)num_clusters - 2.0) * Dpq - nd[p].Sx - nd[q].Sx;
            ++pair_evals;
            if (Qpq < myMin) {
                myMin = Qpq;
                mins.clear();
                mins.push_back({p, q, Qpq});
            } else if (Qpq == myMin) {
                mins.push_back({p, q, Qpq});
            }
        }
        lists.push_back(std::move(mins));
        int idx = (int)lists.size() - 1;
        found[p] = idx;
        return idx;
    }

    // NetMakerOriginal.java:549-561
    double computeRx(int z, int cx, int cy, int num_active) {
        double Rx = 0.0;
        for (int i = 0; i < num_active; ++i) {
            int p = act[i];
            if (p == cx || p == nd[cx].nbr || p == cy || p == nd[cy].nbr || nd[p].nbr < 0)
                Rx += d(z, p);
            else
                Rx += d(z, p) / 2.0;
        }
        return Rx;
    }

    // NeighborNetLocal.java:468-476
    double clusterDistLocal(int p, int u) {
        if (nd[p].nbr < 0) return (d(p, u) + d(p, nd[u].nbr)) / 2.0;
        return (d(p, u) + d(p, nd[u].nbr) + d(nd[p].nbr, u) + d(nd[p].nbr, nd[u].nbr)) / 4.0;
    }

    // NeighborNetLocal.java:388-414
    double agg3wayLocal(int x, int y, int z, int testNode, double subtractedRowSum, int num_clusters, int num_active) {
        double clusterRowSum = 0, clustDistance = 0;
        for (int i = 0; i < num_active; ++i) {
            int p = act[i];
            double myDist = 0;
            if (isRep(p) && (p != x && p != y && p != z)) {
                double Dup = (2.0 / 3.0) * d(x, p) + d(y, p) / 3.0;
                double Dvp = (2.0 / 3.0) * d(z, p) + d(y, p) / 3.0;
                if (nd[p].nbr < 0) {
                    myDist = (Dup + Dvp) / 2.0;
                } else {
                    int pn = nd[p].nbr;
                    double Duq = (2.0 / 3.0) * d(x, pn) + d(y, pn) / 3.0;
                    double Dvq = (2.0 / 3.0) * d(z, pn) + d(y, pn) / 3.0;
                    myDist = (Dup + Dvp + Duq + Dvq) / 4.0;
                }
            }
            if (myDist != 0) clusterRowSum += myDist;
            if (p == testNode) clustDistance = myDist;
        }
        return ((double)num_clusters - 1 - 2.0) * clustDistance - clusterRowSum - (subtractedRowSum + clustDistance);
    }

    // NeighborNetLocal.java:416-466
    double agg4wayLocal(int x2, int x, int y, int y2, int testNode, double subtractedRowSum, int num_clusters, int num_active) {
        std::vector<double> Dup(num_active), Dvp(num_active), Dup2(num_active, 0.0), Dvp2(num_active, 0.0);
        for (int i = 0; i < num_active; ++i) {
            int p = act[i];
            if (p != x) {
                Dup[i] = (2.0 / 3.0) * d(x2, p) + d(x, p) / 3.0;
                Dvp[i] = (2.0 / 3.0) * d(y, p) + d(x, p) / 3.0;
            } else {
                Dup[i] = Dvp[i] = 0;
            }
        }
        double clusterRowSum = 0, clustDistance = 0;
        for (int i = 0; i < num_active; ++i) {
            int p = act[i];
            double myDist = 0;
            if (p != x && p != y && p != y2 && p != x2) {
                if (isRep(p)) {
                    Dup2[i] = (2.0 / 3.0) * Dup[i] + Dvp[i] / 3.0;
                    Dvp2[i] = (2.0 / 3.0) * d(y2, p) + Dvp[i] / 3.0;
                    if (nd[p].nbr < 0) {
                        myDist = (Dup2[i] + Dvp2[i]) / 2.0;
                    } else {
                        int j = nd[nd[p].nbr].pos;
                        Dup2[j] = (2.0 / 3.0) * Dup[j] + Dvp[j] / 3.0;
                        Dvp2[j] = (2.0 / 3.0) * d(y2, nd[p].nbr) + Dvp[j] / 3.0;
                        myDist = (Dup2[i] + Dvp2[i] + Dup2[j] + Dvp2[j]) / 4.0;
                    }
                }
            } else {
                Dup2[i] = Dvp2[i] = 0;
            }
            clusterRowSum += myDist;
            if (p == testNode) clustDistance = myDist;
        }
        return ((double)num_clusters - 1 - 2.0) * clustDistance - clusterRowSum - (subtractedRowSum + clustDistance);
    }

    // the 4-candidate pick shared by NetMakerOriginal.java:409-452 and
    // NeighborNetLocal.java:292-335
    void pickXY(int cx, int cy, int num_active, int num_clusters, int& x, int& y) {
        x = cx; y = cy;
        double Cx_Rx = 0.0, Cx_nbr_Rx = 0.0, Cy_Rx = 0.0, Cy_nbr_Rx = 0.0;
        int cxn = nd[cx].nbr, cyn = nd[cy].nbr;
        if (cxn >= 0 || cyn >= 0) {
            Cx_Rx = computeRx(cx, cx, cy, num_active);
            if (cxn >= 0) Cx_nbr_Rx = computeRx(cxn, cx, cy, num_active);
            Cy_Rx = computeRx(cy, cx, cy, num_active);
            if (cyn >= 0) Cy_nbr_Rx = computeRx(cyn, cx, cy, num_active);
        }
        int m = num_clusters;
        if (cxn >= 0) m++;
        if (cyn >= 0) m++;
        best = ((double)m - 2.0) * d(cx, cy) - Cx_Rx - Cy_Rx;
        if (cxn >= 0) {
            double Q = ((double)m - 2.0) * d(cxn, cy) - Cx_nbr_Rx - Cy_Rx;
            if (Q < best) { x = cxn; y = cy; best = Q; }
        }
        if (cyn >= 0) {
            double Q = ((double)m - 2.0) * d(cx, cyn) - Cx_Rx - Cy_nbr_Rx;
            if (Q < best) { x = cx; y = cyn; best = Q; }
        }
        if (cxn >= 0 && cyn >= 0) {
            double Q = ((double)m - 2.0) * d(cxn, cyn) - Cx_nbr_Rx - Cy_nbr_Rx;
            if (Q < best) { x = cxn; y = cyn; best = Q; }
        }
    }

    // NeighborNetLocal.java:280-386
    double findAgglomeratedQ(int cx, int cy, int testNode, int num_clusters, int num_active) {
        int x, y;
        pickXY(cx, cy, num_active, num_clusters, x, y);
        double subtractedRowSum = nd[testNode].Sx - clusterDist(cx, testNode) - clusterDist(cy, testNode);
        if (nd[x].nbr < 0 && nd[y].nbr < 0) {
            // NeighborNetLocal.java:349: calculateClusterDistLocal(x, testNode) dereferences
            // testNode.nbr; when testNode is a singleton the JVM throws (F7-class bug).  With a
            // singleton test node we fall back to the 2-term form against (x,y), which is what
            // the loop at :351-360 computes for that same node.
            double Dpu;
            if (nd[testNode].nbr >= 0) Dpu = clusterDistLocal(x, testNode);
            else { Dpu = (d(testNode, x) + d(testNode, y)) / 2.0; ++npe_would_fire; }
            double clusterRowSum = 0;
            for (int i = 0; i < num_active; ++i) {
                int p = act[i];
                if (isRep(p) && (p != x && p != y)) {
                    if (nd[p].nbr < 0) clusterRowSum += (d(p, x) + d(p, y)) / 2.0;
                    else clusterRowSum += (d(p, x) + d(p, y) + d(nd[p].nbr, x) + d(nd[p].nbr, y)) / 4.0;
                }
            }
            return ((double)num_clusters - 1 - 2.0) * Dpu - clusterRowSum - (subtractedRowSum + Dpu);
        } else if (nd[x].nbr < 0) {
            return agg3wayLocal(x, y, nd[y].nbr, testNode, subtractedRowSum, num_clusters, num_active);
        } else if (nd[y].nbr < 0 || num_active == 4) {
            return agg3wayLocal(y, x, nd[x].nbr, testNode, subtractedRowSum, num_clusters, num_active);
        } else {
            return agg4wayLocal(nd[x].nbr, x, y, nd[y].nbr, testNode, subtractedRowSum, num_clusters, num_active);
        }
    }

    // NeighborNetLocal.java:170-264
    void findNodesRelaxed(int num_active, int num_clusters) {
        RowCache found;
        lists.clear();
        std::vector<RowMin> myMinimums;
        if (firstTime) {
            rowPerm.resize(n);
            for (int i = 0; i < n; ++i) rowPerm[i] = i;
            firstTime = false;
            top = (int)n - 1;
        }
        for (int i = top + 1; i > 0; i--) {
            int swapCell = rng.nextInt(i);
            if (rowPerm[swapCell] >= num_active) {
                std::swap(rowPerm[swapCell], rowPerm[top]);
                if (i == top + 1) i--; else i++;
                top--;
                continue;
            }
            std::swap(rowPerm[i - 1], rowPerm[swapCell]);
            int p = act[rowPerm[i - 1]];
            if (nd[p].nbr >= 0 && nd[nd[p].nbr].id < nd[p].id) continue;
            int li = findRowMin(p, found, num_active, num_clusters);
            // lists may reallocate inside the inner findRowMin: index, don't hold references
            for (size_t a = 0; a < lists[li].size(); ++a) {
                RowMin myRM = lists[li][a];
                int lo = findRowMin(myRM.row, found, num_active, num_clusters);
                for (size_t b = 0; b < lists[lo].size(); ++b) {
                    RowMin t = lists[lo][b];
                    int rn = nd[t.row].nbr, pn = nd[p].nbr;
                    if ((t.row == p) || (rn >= 0 && rn == p) || (rn >= 0 && pn >= 0 && rn == pn) || (pn >= 0 && t.row == pn)) {
                        myMinimums.push_back(t);
                        break;
                    }
                }
            }
            if (!myMinimums.empty()) {
                int choice = rng.nextInt((int)myMinimums.size());
                RowMin c = myMinimums[choice];
                Cx = c.me; Cy = c.row;
                if (additive) {
                    // The reference loops `choice = (choice+1) % max` until it is back at `initial` (:226-255), but it
                    // never re-reads combineMe, so every pass repeats the IDENTICAL test on the same (Cx, Cy): the
                    // outcome of the first pass is the outcome of the loop.  Evaluate once (the literal loop costs
                    // myMinimums.size() identical O(m) look-aheads and myMinimums is never cleared, :172).
                    bool accepted = false;
                    {
                        // INTENDED test-node loop (documented deviation, SURVEY F7): the shipped
                        // `for (int j = num_active-1; i > 0; i--)` never moves j and NPEs when
                        // netNodes[num_active-1] lies in the two clusters.
                        int testNode = -1;
                        int j = num_active - 1;
                        if (act[j] == Cx || act[j] == Cy || act[j] == nd[Cx].nbr || act[j] == nd[Cy].nbr) ++npe_would_fire;
                        for (; j >= 0; j--) {
                            int t = act[j];
                            if (t == Cx || t == Cy || t == nd[Cx].nbr || t == nd[Cy].nbr) continue;
                            testNode = t; break;
                        }
                        if (testNode < 0) accepted = true;   // nothing outside the two clusters
                        else {
                            if (nd[testNode].nbr >= 0 && nd[nd[testNode].nbr].id < nd[testNode].id) testNode = nd[testNode].nbr;
                            double originalDistCx = clusterDist(Cx, testNode);
                            double originalQ = ((double)num_clusters - 2.0) * originalDistCx - nd[Cx].Sx - nd[testNode].Sx;
                            double newQ = findAgglomeratedQ(Cx, Cy, testNode, num_clusters, num_active);
                            if (std::fabs(originalQ - newQ) < .0000001) accepted = true;
                        }
                    }
                    if (accepted) return;
                } else {
                    return;
                }
            }
        }
    }

    // ---- Relaxed, driven by the product's state machine (fnn_relaxed_sm.h) with CPU row scans ----------------
    relaxed::Machine SM{};
    std::vector<int> sm_rowPerm, sm_epoch, sm_clist, sm_loff, sm_lcnt, sm_lme, sm_tie, sm_mymin;
    bool sm_init = false;
    struct SMView {
        Engine* e; int num_active;
        int m() const { return num_active; }
        int id_at(int pos) const { return e->nd[e->act[pos]].id; }
        int nbr_pos(int pos) const { int h = e->nd[e->act[pos]].nbr; return h < 0 ? -1 : e->nd[h].pos; }
    };
    void findNodesRelaxedSM(int num_active, int num_clusters) {
        if (!sm_init) {
            sm_rowPerm.assign(n, 0); sm_epoch.assign(n, 0); sm_clist.assign(n, 0);
            sm_loff.assign(2 * n + 16, 0); sm_lcnt.assign(2 * n + 16, 0); sm_lme.assign(2 * n + 16, 0);
            sm_tie.assign(16 * n + 65536, 0); sm_mymin.assign(2 * (8 * n + 65536), 0);
            SM.rng = rng.s; SM.top = 0; SM.first_time = 1;
            SM.rowPerm = sm_rowPerm.data(); SM.cache_epoch = sm_epoch.data(); SM.cache_list = sm_clist.data();
            SM.list_off = sm_loff.data(); SM.list_cnt = sm_lcnt.data(); SM.list_me = sm_lme.data();
            SM.tiepool = sm_tie.data(); SM.mymin = sm_mymin.data();
            SM.max_lists = (int)sm_loff.size(); SM.tie_cap = (int)sm_tie.size(); SM.mymin_cap = (int)sm_mymin.size() / 2;
            SM.epoch = 0; SM.additive = additive ? 1 : 0; SM.cx_pos = SM.cy_pos = -1;
            sm_init = true;
        }
        SMView nv{this, num_active};
        relaxed::begin_call(SM, (int)n);
        int look_accept = 0;
        int nscan = 0;
        while (true) {
            const relaxed::Request rq = relaxed::step(SM, nv, look_accept);
            if (rq == relaxed::REQ_DONE) break;
            if (rq == relaxed::REQ_ERROR) { status = -11; break; }
            if (rq == relaxed::REQ_SCAN) {
                const int p = act[SM.req_pos];
                double myMin = 1.7976931348623157e308;
                int cnt = 0;
                int* out = SM.tiepool + SM.tie_used;
                const int room = relaxed::tie_room(SM);
                for (int row = 0; row < num_active; ++row) {
                    const int q = act[row];
                    if (p == q || (nd[p].nbr >= 0 && nd[p].nbr == q)) continue;
                    const double Qpq = ((double)num_clusters - 2.0) * clusterDist(p, q) - nd[p].Sx - nd[q].Sx;
                    ++pair_evals;
                    if (Qpq < myMin) { myMin = Qpq; cnt = 0; if (cnt < room) out[cnt] = row; cnt = 1; }
                    else if (Qpq == myMin) { if (cnt < room) out[cnt] = row; ++cnt; }
                }
                if (rec_row) {   // scans, ties, digest of fnn_record.h
                    uint64_t dg = rec::scan_term(nscan, SM.req_pos, -1, 0);
                    for (int r = 0; r < cnt && r < room; ++r) dg += rec::scan_term(nscan, SM.req_pos, r, out[r]);
                    rec_row[0] += 1; rec_row[1] += cnt;
                    rec_row[3] = (int64_t)((uint64_t)rec_row[3] + dg);
                }
                ++nscan;
                if (cnt > room || !relaxed::commit_scan(SM, cnt)) { status = -12; break; }
            } else {   // REQ_LOOKAHEAD
                if (rec_row) rec_row[2] += 1;
                const int cx = act[SM.cx_pos], cy = act[SM.cy_pos], t = act[SM.look_test_pos];
                const double originalQ = ((double)num_clusters - 2.0) * clusterDist(cx, t) - nd[cx].Sx - nd[t].Sx;
                const double newQ = findAgglomeratedQ(cx, cy, t, num_clusters, num_active);
                look_accept = std::fabs(originalQ - newQ) < .0000001;
            }
        }
        if (SM.cx_pos >= 0 && SM.cy_pos >= 0) { Cx = act[SM.cx_pos]; Cy = act[SM.cy_pos]; }
    }

    // ---- Random (NeighborNetRandom.java) -----------------------------------
    // :31-48
    int64_t findSearchAmount(int total) {
        int64_t amount;
        switch (mode) {
            case RANDOM_LOGN: amount = (int64_t)std::ceil(std::log10((double)total)); break;
            case RANDOM_N: amount = total; break;
            default: amount = (int64_t)std::ceil(std::log10((double)total)) * (int64_t)total; break;
        }
        return (int64_t)mult * amount;
    }
    // :130-178 (numThreads == 1 branch)
    void findNodesRandom(int num_active, int num_clusters) {
        best = 1.7976931348623157e308;
        const int64_t searchAmount = findSearchAmount(num_active);
        int i = rng.nextInt(num_active);
        int j;
        Cx = Cy = -1;
        if (rec_row) rec_row[0] = searchAmount;
        for (int64_t k = 0; k < searchAmount; ++k) {
            const uint64_t one_step = (rng.s * 0x5DEECE66DULL + 0xBULL) & ((1ULL << 48) - 1);
            int j0;
            if (nd[act[i]].nbr >= 0) {
                int iNbr = nd[nd[act[i]].nbr].pos;
                j = j0 = rng.nextInt(num_active - 2);
                if (i == j && num_active - 1 == iNbr) j = num_active - 2;
                else if (i == j && num_active - 1 != iNbr) j = num_active - 1;
                else if (iNbr == j && num_active - 2 == i) j = num_active - 1;
                else if (iNbr == j && num_active - 2 != i) j = num_active - 2;
            } else {
                j = j0 = rng.nextInt(num_active - 1);
                if (i == j) j = num_active - 1;
            }
            if (rec_row) {   // nextInt rejected (took more than one LCG step); remapped; digest of fnn_record.h
                rec_row[1] += rng.s != one_step;
                rec_row[2] += j != j0;
                rec_row[3] = (int64_t)((uint64_t)rec_row[3] + rec::draw_term(k, i, j));
            }
            int p = act[i], q = act[j];
            double Dpq = clusterDist(p, q);
            double Qpq = ((double)num_clusters - 2.0) * Dpq - nd[p].Sx - nd[q].Sx;
            ++pair_evals;
            if ((Cx < 0 || (Qpq < best)) && (nd[p].nbr != q)) { Cx = p; Cy = q; best = Qpq; }
            i = j;
        }
    }

    // ---- reduction ----------------------------------------------------------
    // NetMakerOriginal.java:681-696
    void subtractClusterDistance(int p, int x) {
        if (p != x && p != nd[x].nbr && isRep(p)) {
            double Dpx = clusterDist(p, x);
            nd[p].Sx -= Dpx;
            if (nd[p].nbr >= 0) nd[nd[p].nbr].Sx -= Dpx;
        }
    }
    // :570-577
    int agg2way(int x, int y) { nd[x].nbr = y; nd[y].nbr = x; return x; }
    // :589-674
    int agg3way(int x, int y, int z, int num_nodes, int num_active) {
        Node U; U.id = num_nodes + 1; U.ch1 = x; U.ch2 = y;
        Node V; V.id = num_nodes + 2; V.ch1 = y; V.ch2 = z;
        nd.push_back(U); int u = (int)nd.size() - 1;
        nd.push_back(V); int v = (int)nd.size() - 1;
        act[nd[x].pos] = u; nd[u].pos = nd[x].pos; nd[u].dist = nd[x].dist;
        act[nd[z].pos] = v; nd[v].pos = nd[z].pos; nd[v].dist = nd[z].dist;
        act[nd[y].pos] = act[num_active - 1];
        nd[act[nd[y].pos]].pos = nd[y].pos;
        act[num_active - 1] = -1;
        nd[u].nbr = v; nd[v].nbr = u;
        for (int i = 0; i < num_active - 1; ++i) {
            int p = act[i];
            double t1 = (2.0 / 3.0) * d(x, p) + d(y, p) / 3.0;
            d(p, u) = t1; d(u, p) = t1;
            double t2 = (2.0 / 3.0) * d(z, p) + d(y, p) / 3.0;
            d(p, v) = t2; d(v, p) = t2;
        }
        d(v, v) = 0.0; d(u, u) = 0.0;
        stack.push_back(u);
        return u;
    }
    // :707-726
    int agg4way(int x2, int x, int y, int y2, int num_nodes, int num_active) {
        int u = agg3way(x2, x, y, num_nodes, num_active);
        num_nodes += 2;
        int v = agg3way(u, nd[u].nbr, y2, num_nodes, num_active - 1);
        nd[x2].pos = -1; nd[x].pos = -1; nd[y].pos = -1; nd[y2].pos = -1;
        nd[u].pos = -1; nd[nd[u].nbr].pos = -1;
        return v;
    }
    // :517-536
    void updateClusterDistances(int u, int num_active) {
        nd[u].Sx = 0; nd[nd[u].nbr].Sx = 0;
        for (int i = 0; i < num_active; ++i) {
            int p = act[i];
            if (isRep(p) && nd[u].nbr != p && u != p) {
                double Dpu = clusterDistLocal(p, u);
                nd[p].Sx += Dpu;
                if (nd[p].nbr >= 0) nd[nd[p].nbr].Sx += Dpu;
                nd[u].Sx += Dpu;
            }
        }
        nd[nd[u].nbr].Sx = nd[u].Sx;
    }

    // NetMakerOriginal.java:397-515
    void handleAgglomerationEvent(int cx, int cy, int& num_nodes, int& num_active, int& num_clusters, TraceRow& tr) {
        int x, y;
        pickXY(cx, cy, num_active, num_clusters, x, y);
        tr.x_id = nd[x].id; tr.y_id = nd[y].id; tr.best = best;
        for (int i = 0; i < num_active; ++i) {
            int p = act[i];
            if (i != nd[x].pos && i != nd[y].pos) {
                subtractClusterDistance(p, x);
                subtractClusterDistance(p, y);
            }
        }
        int u;
        if (nd[x].nbr < 0 && nd[y].nbr < 0) {
            u = agg2way(x, y);
            num_clusters--;
            tr.kind = 2;
        } else if (nd[x].nbr < 0) {
            int yn = nd[y].nbr;
            u = agg3way(x, y, yn, num_nodes, num_active);
            num_nodes += 2; num_active--; num_clusters--;
            nd[x].pos = -1; nd[y].pos = -1; nd[yn].pos = -1;
            tr.kind = 3;
        } else if (nd[y].nbr < 0 || num_active == 4) {
            int xn = nd[x].nbr;
            u = agg3way(y, x, xn, num_nodes, num_active);
            num_nodes += 2; num_active--; num_clusters--;
            nd[x].pos = -1; nd[y].pos = -1; nd[xn].pos = -1;
            tr.kind = 3;
        } else {
            u = agg4way(nd[x].nbr, x, y, nd[y].nbr, num_nodes, num_active);
            num_nodes += 4; num_active -= 2; num_clusters--;
            tr.kind = 4;
        }
        updateClusterDistances(u, num_active);
    }

    // NetMakerOriginal.java:331-395
    int agglomNodes(int num_nodes) {
        int num_active = num_nodes, num_clusters = num_nodes;
        for (int64_t iter = 0; num_active > 3; ++iter) {
            if (max_iters > 0 && iter >= max_iters) { stopped = true; break; }
            if (record) {   // a zero row unless the strategy runs in this iteration
                record->insert(record->end(), rec::COLS, 0);
                rec_row = record->data() + record->size() - rec::COLS;
            }
            if (num_active == 4 && num_clusters == 2) {
                int p = act[0];
                int q = (nd[p].nbr != act[1]) ? act[1] : act[2];
                TraceRow tr{num_active, num_clusters, nd[p].id, nd[q].id, 0, 0, 5, 0.0};
                if (d(p, q) + d(nd[p].nbr, nd[q].nbr) < d(p, nd[q].nbr) + d(nd[p].nbr, q)) {
                    agg3way(p, q, nd[q].nbr, num_nodes, num_active);
                    num_nodes += 2;
                    tr.x_id = nd[q].id;
                } else {
                    agg3way(p, nd[q].nbr, q, num_nodes, num_active);
                    num_nodes += 2;
                    tr.x_id = nd[nd[q].nbr].id;
                }
                if (trace) trace->push_back(tr);
                break;
            }
            if (mode == CANONICAL || num_active <= fallback) {
                int pairs = 0;
                for (int i = 0; i < num_active; ++i) if (nd[act[i]].nbr >= 0) ++pairs;
                alg_bytes += 4.0 * (double)num_active * ((double)num_active - 1.0) - 4.0 * (double)pairs + 8.0 * (double)num_active;
            }
            if (mode == CANONICAL && threads > 1 && num_active > fallback) findNodesCanonicalMT(num_active, num_clusters);
            else if (num_active <= fallback || mode == CANONICAL) findNodesDefault(num_active, num_clusters);
            else if (mode == RELAXED && g_use_relaxed_sm) findNodesRelaxedSM(num_active, num_clusters);
            else if (mode == RELAXED) findNodesRelaxed(num_active, num_clusters);
            else findNodesRandom(num_active, num_clusters);
            if (Cx < 0 || Cy < 0) { status = -10; return num_nodes; }
            if (nd[Cx].id > nd[Cy].id) std::swap(Cx, Cy);
            TraceRow tr{num_active, num_clusters, nd[Cx].id, nd[Cy].id, 0, 0, 0, 0.0};
            handleAgglomerationEvent(Cx, Cy, num_nodes, num_active, num_clusters, tr);
            if (trace) trace->push_back(tr);
        }
        return num_nodes;
    }

    // NetMakerOriginal.java:246-325
    void expandNodes(int32_t* ordering) {
        int x = act[0], y = act[1], z = act[2];
        nd[x].next = y; nd[y].next = z; nd[z].next = x;
        nd[x].prev = z; nd[y].prev = x; nd[z].prev = y;
        while (!stack.empty()) {
            int u = stack.back(); stack.pop_back();
            int v = nd[u].nbr;
            x = nd[u].ch1; y = nd[u].ch2; z = nd[v].ch2;
            if (v != nd[u].next) {
                std::swap(u, v);
                std::swap(x, z);
            }
            nd[x].prev = nd[u].prev;
            nd[nd[x].prev].next = x;
            nd[x].next = y; nd[y].prev = x;
            nd[y].next = z; nd[z].prev = y;
            nd[z].next = nd[v].next;
            nd[nd[z].next].prev = z;
        }
        while (nd[x].id != 1) x = nd[x].next;
        int a = x, t = 0;
        ordering[0] = 0;
        do { ordering[++t] = nd[a].id; a = nd[a].next; } while (a != x);
    }

    // NetMakerOriginal.java:129-162
    int run(int32_t* ordering) {
        if (n <= 3) { for (int i = 0; i <= n; ++i) ordering[i] = i; return 0; }
        nd.reserve(3 * n + 8);
        nd.resize(n);
        act.assign(n, -1);
        for (int i = (int)n; i >= 1; --i) {
            Node& t = nd[i - 1];
            t.id = i; t.pos = i - 1; t.dist = i - 1;
            act[i - 1] = i - 1;
        }
        initialize((int)n);
        agglomNodes((int)n);
        if (status != 0) return status;
        if (stopped) { for (int64_t i = 0; i <= n; ++i) ordering[i] = 0; return 0; }
        expandNodes(ordering);
        return 0;
    }
};

// ---- CircularSplitWeights.java, literal (parity ladder level L0) -----------
// :247-271
void unconstrainedLS(int64_t n, const double* d, double* x) {
    int64_t index = 0;
    for (int64_t i = 0; i <= n - 3; i++) {
        x[index] = (d[index] + d[index + (n - i - 2) + 1] - d[index + 1]) / 2.0;
        index++;
        for (int64_t j = i + 2; j <= n - 2; j++) {
            x[index] = (d[index] + d[index + (n - i - 2) + 1] - d[index + 1] - d[index + (n - i - 2)]) / 2.0;
            index++;
        }
        if (i == 0) x[index] = (d[0] + d[n - 2] - d[2 * n - 4]) / 2.0;
        else x[index] = (d[index] + d[i] - d[i - 1] - d[index + (n - i - 2)]) / 2.0;
        index++;
    }
    x[index] = (d[index] + d[n - 2] - d[n - 3]) / 2.0;
}
// :571-591
double rowsum(int64_t n, const double* d, int64_t k) {
    double r = 0;
    int64_t index = 0;
    if (k > 0) {
        index = k - 1;
        for (int64_t i = 0; i < k; i++) { r += d[index]; index += (n - i - 2); }
        index++;
    }
    for (int64_t j = k + 1; j < n; j++) r += d[index++];
    return r;
}
// :603-633
void calcAtx(int64_t n, const double* d, double* p) {
    int64_t index = 0;
    for (int64_t i = 0; i < n - 1; i++) { p[index] = rowsum(n, d, i + 1); index += (n - i - 1); }
    index = 1;
    for (int64_t i = 0; i < n - 2; i++) {
        p[index] = p[index - 1] + p[index + (n - i - 2)] - 2 * d[index + (n - i - 2)];
        index += (n - i - 2) + 1;
    }
    for (int64_t k = 3; k <= n - 1; k++) {
        index = k - 1;
        for (int64_t i = 0; i <= n - k - 1; i++) {
            p[index] = p[index - 1] + p[index + n - i - 2] - p[index + n - i - 3] - 2.0 * d[index + n - i - 2];
            index += (n - i - 2) + 1;
        }
    }
}
// :643-731
void calcAb(int64_t n, const double* b, double* d) {
    int64_t index, dindex = 0;
    for (int64_t i = 0; i <= n - 2; i++) {
        double d_ij = 0.0;
        index = i - 1;
        for (int64_t k = 0; k <= i - 1; k++) { d_ij += b[index]; index += (n - k - 2); }
        index++;
        for (int64_t k = i + 1; k <= n - 1; k++) d_ij += b[index++];
        d[dindex] = d_ij;
        dindex += (n - i - 2) + 1;
    }
    index = 1;
    for (int64_t i = 0; i <= n - 3; i++) {
        d[index] = d[index - 1] + d[index + (n - i - 2)] - 2 * b[index - 1];
        index += 1 + (n - i - 2);
    }
    for (int64_t k = 3; k <= n - 1; k++) {
        index = k - 1;
        for (int64_t i = 0; i <= n - k - 1; i++) {
            d[index] = d[index - 1] + d[index + (n - i - 2)] - d[index + (n - i - 2) - 1] - 2.0 * b[index - 1];
            index += 1 + (n - i - 2);
        }
    }
}
// :740-749
double normsq(const double* x, int64_t n) {
    double ss = 0.0;
    for (int64_t k = 0; k < n; k++) { double xk = x[k]; ss += xk * xk; }
    return ss;
}
struct CswStats { int64_t cg_iters = 0, cg_calls = 0, outer = 0, inner = 0; };
// :769-831
void conjugateGrads(int64_t ntax, int64_t npairs, double* r, double* w, double* p, double* y,
                    const double* W, const double* b, const uint8_t* active, double* x, int64_t kmax, CswStats& st) {
    st.cg_calls++;
    calcAb(ntax, x, y);
    for (int64_t k = 0; k < npairs; k++) y[k] = W[k] * y[k];
    calcAtx(ntax, y, r);
    for (int64_t k = 0; k < npairs; k++) r[k] = active[k] ? 0.0 : b[k] - r[k];
    double rho = normsq(r, npairs), rho_old = 0;
    double e_0 = 1e-8 * std::sqrt(normsq(b, npairs));
    int64_t k = 0;
    while ((rho > e_0 * e_0) && (k < kmax)) {
        k = k + 1;
        st.cg_iters++;
        if (k == 1) { for (int64_t i = 0; i < npairs; i++) p[i] = r[i]; }
        else { double beta = rho / rho_old; for (int64_t i = 0; i < npairs; i++) p[i] = r[i] + beta * p[i]; }
        calcAb(ntax, p, y);
        for (int64_t i = 0; i < npairs; i++) y[i] *= W[i];
        calcAtx(ntax, y, w);
        for (int64_t i = 0; i < npairs; i++) if (active[i]) w[i] = 0.0;
        double alpha = 0.0;
        for (int64_t i = 0; i < npairs; i++) alpha += p[i] * w[i];
        alpha = rho / alpha;
        for (int64_t i = 0; i < npairs; i++) { x[i] += alpha * p[i]; r[i] -= alpha * w[i]; }
        rho_old = rho;
        rho = normsq(r, npairs);
    }
}
// :282-330
bool worstIndices(const double* x, int64_t n, double propKept, std::vector<int64_t>& result) {
    result.clear();
    if (propKept == 0) return false;
    int64_t numNeg = 0;
    for (int64_t i = 0; i < n; i++) if (x[i] < 0.0) numNeg++;
    if (numNeg == 0) return false;
    std::vector<double> xc; xc.reserve(numNeg);
    for (int64_t i = 0; i < n; i++) if (x[i] < 0.0) xc.push_back(x[i]);
    std::sort(xc.begin(), xc.end());
    int64_t nkept = (int64_t)std::ceil(propKept * (double)numNeg);
    double cutoff = xc[nkept - 1];
    result.assign(nkept, 0);
    int64_t front = 0, back = nkept - 1;
    for (int64_t i = 0; i < n; i++) {
        if (x[i] < cutoff) result[front++] = i;
        else if (x[i] == cutoff) { if (back >= front) result[back--] = i; }
    }
    return true;
}
// :359-557 (diagnostic prints dropped).  kmax: iteration cap of every CG call (npairs in the reference, :774);
// max_cg_calls > 0: return right after that many CG calls (the budget of fnn_split_weights_budget).
void activeConjugate(int64_t ntax, int64_t npairs, const double* d, const double* W, double* x, std::vector<uint8_t>& active,
                     int64_t kmax, int64_t max_cg_calls, CswStats& st) {
    unconstrainedLS(ntax, d, x);
    bool all_positive = true;
    for (int64_t k = 0; k < npairs && all_positive; k++) if (x[k] < 0.0) all_positive = false;
    if (all_positive) return;
    std::vector<double> r(npairs), w(npairs), p(npairs), y(npairs), old_x(npairs, 1.0), AtWd(npairs);
    for (int64_t k = 0; k < npairs; k++) y[k] = W[k] * d[k];
    calcAtx(ntax, y.data(), AtWd.data());
    bool first_pass = true;
    std::vector<int64_t> contract;
    auto cg = [&]() {
        conjugateGrads(ntax, npairs, r.data(), w.data(), p.data(), y.data(), W, AtWd.data(), active.data(), x, kmax, st);
        return max_cg_calls > 0 && st.cg_calls >= max_cg_calls;   // budget spent
    };
    while (true) {
        st.outer++;
        while (true) {
            st.inner++;
            if (!first_pass && cg()) return;
            first_pass = false;
            if (worstIndices(x, npairs, 0.6, contract)) {
                for (int64_t idx : contract) { x[idx] = 0.0; active[idx] = 1; }
                if (cg()) return;
            }
            int64_t min_i = -1; double min_xi = -1.0;
            for (int64_t i = 0; i < npairs; i++) {
                if (x[i] < 0.0) {
                    double xi = (old_x[i]) / (old_x[i] - x[i]);
                    if ((min_i == -1) || (xi < min_xi)) { min_i = i; min_xi = xi; }
                }
            }
            if (min_i == -1) break;
            for (int64_t i = 0; i < npairs; i++) if (!active[i]) old_x[i] += min_xi * (x[i] - old_x[i]);
            active[min_i] = 1;
            x[min_i] = 0.0;
        }
        calcAb(ntax, x, y.data());
        for (int64_t i = 0; i < npairs; i++) y[i] *= W[i];
        calcAtx(ntax, y.data(), r.data());
        int64_t min_i = -1; double min_grad = 1.0;
        for (int64_t i = 0; i < npairs; i++) {
            r[i] -= AtWd[i];
            r[i] *= 2.0;
            if (active[i]) {
                double g = r[i];
                if ((min_i == -1) || (g < min_grad)) { min_i = i; min_grad = g; }
            }
        }
        if ((min_i == -1) || (min_grad > -0.0000001)) return;
        active[min_i] = 0;
    }
}

inline int64_t upperIndex(int64_t n, int64_t i, int64_t j) {   // DistancesAndNames.java:24-38
    if (j < i) std::swap(i, j);
    return i * (n - 1) - i * (i - 1) / 2 + j - (i + 1);
}

}  // namespace

extern "C" {

// 1: Relaxed findNodes runs through the product's state machine (fnn_relaxed_sm.h) instead of the literal restatement
void oracle_set_relaxed_sm(int on) { g_use_relaxed_sm = on; }

// Ordering.  D is n*n row-major and is mutated in place (like the Java double[][]).
// trace_out: optional [max_trace][8] doubles (m,c,cx,cy,x,y,kind,best); returns rows in *n_trace.
// record_out: optional [max_trace][4] int64, the strategy record of fnn_ctx_strategy_record (Relaxed: only through the
// product's state machine, oracle_set_relaxed_sm(1), whose scan sequence is the device's); requires trace_out.
// max_iters > 0: stop after that many agglomeration iterations and return the trace so far (a prefix of the full trace);
// the ordering is then all zeros.  0 = run to the end.
int oracle_order(int mode, int64_t n, double* D, int64_t seed, int mult, int additive, int fallback,
                 int32_t* ordering, double* trace_out, int64_t max_trace, int64_t* n_trace,
                 int64_t* counters /* [0]=pair_evals [1]=npe_would_fire */, int threads, double* alg_bytes,
                 int64_t max_iters, int64_t* record_out) {
    Engine e;
    e.n = n; e.D = D; e.mode = mode; e.mult = mult; e.additive = additive != 0; e.fallback = fallback;
    e.max_iters = max_iters;
    e.rng = JavaRandom(seed);
    e.threads = threads < 1 ? 1 : threads;
    std::vector<TraceRow> tr;
    if (trace_out) e.trace = &tr;
    std::vector<int64_t> rc_rows;
    if (record_out) e.record = &rc_rows;
    int rc = e.run(ordering);
    if (record_out) {   // one row per trace row (the record is only kept together with the trace)
        const int64_t k = std::min<int64_t>((int64_t)rc_rows.size() / rec::COLS, max_trace);
        std::copy(rc_rows.begin(), rc_rows.begin() + rec::COLS * k, record_out);
    }
    if (trace_out) {
        int64_t k = std::min<int64_t>((int64_t)tr.size(), max_trace);
        for (int64_t i = 0; i < k; ++i) {
            double* o = trace_out + 8 * i;
            o[0] = tr[i].m; o[1] = tr[i].c; o[2] = tr[i].cx_id; o[3] = tr[i].cy_id;
            o[4] = tr[i].x_id; o[5] = tr[i].y_id; o[6] = tr[i].kind; o[7] = tr[i].best;
        }
        if (n_trace) *n_trace = (int64_t)tr.size();
    }
    if (counters) { counters[0] = e.pair_evals; counters[1] = e.npe_would_fire; }
    if (alg_bytes) *alg_bytes = e.alg_bytes;
    return rc;
}

// initial row sums only (NetMakerOriginal.java:164-191), for kernel K1 tests
void oracle_rowsums(int64_t n, const double* D, double* Sx) {
    for (int64_t k = 0; k < n; ++k) {
        double s = 0.0;
        for (int64_t j = 0; j < n; ++j) if (j != k) s += D[k * n + j];
        Sx[k] = s;
    }
}

// d in circular-position order from file-order packed upper triangle, with the
// ROTATED permutation (SURVEY F4): position 0 <-> ordering[n], position p <-> ordering[p].
void oracle_setup_d(int64_t n, const int32_t* ordering, const double* d_upper, double* d_pos) {
    int64_t idx = 0;
    for (int64_t i = 0; i < n; ++i)
        for (int64_t j = i + 1; j < n; ++j) {
            int64_t ti = (i == 0 ? ordering[n] : ordering[i]) - 1;
            int64_t tj = ordering[j] - 1;
            d_pos[idx++] = d_upper[upperIndex(n, ti, tj)];
        }
}

void oracle_unconstrained_ls(int64_t n, const double* d, double* x) { unconstrainedLS(n, d, x); }
void oracle_atx(int64_t n, const double* d, double* p) { calcAtx(n, d, p); }
void oracle_ab(int64_t n, const double* b, double* d) { calcAb(n, b, d); }

// CircularSplitWeights.getWeights (:162-189) with var="ols" (W == 1), constrained.
// d_pos: distances already in circular-position order (oracle_setup_d).  max_cg_iters / max_cg_calls: the budget of
// fnn_split_weights_budget (include/fastnn.h), 0 = none.  active_out (optional, npairs bytes): 1 = split held at zero by the
// active set when the solver returned.
int oracle_split_weights(int64_t n, const double* d_pos, double* x, int constrained, int64_t* stats /*[4]*/, int64_t max_cg_iters,
                         int64_t max_cg_calls, uint8_t* active_out) {
    int64_t npairs = n * (n - 1) / 2;
    CswStats st;
    std::vector<uint8_t> active(npairs, 0);
    if (!constrained) unconstrainedLS(n, d_pos, x);
    else {
        std::vector<double> W(npairs, 1.0);   // v filled 1.0, W = 1/v (:172-177, :213-236)
        activeConjugate(n, npairs, d_pos, W.data(), x, active, max_cg_iters > 0 ? std::min(npairs, max_cg_iters) : npairs,
                        max_cg_calls, st);
    }
    if (active_out) std::copy(active.begin(), active.end(), active_out);
    if (stats) { stats[0] = st.cg_iters; stats[1] = st.cg_calls; stats[2] = st.outer; stats[3] = st.inner; }
    return 0;
}

// java.util.Random stream, for pinning the LCG against published known answers
// The PRODUCT's tile sequence / multi-GPU partition (csrc/fnn_tile_iter.h), compiled for the host so that the CPU (gloo)
// tests of the N>1 path exercise the kernels' own code, not a mirror: tiles of CTA `cta` of rank `rank` (world ranks,
// `grid` CTAs per rank) for m active nodes -> (first row, first column) pairs; returns the count (or the count needed).
int64_t oracle_tile_sequence(int m, int rank, int world, int cta, int grid, int32_t* r0_out, int32_t* c0_out, int64_t cap) {
    int64_t k = 0;
    for (tma::TileIter it(m, rank + world * cta, world * grid); it.valid(); it.next()) {
        int r0, c0;
        it.decode(r0, c0);
        if (k < cap) { r0_out[k] = r0; c0_out[k] = c0; }
        ++k;
    }
    return k;
}
int oracle_tile_rows(void) { return tma::TILE_ROWS; }
int oracle_tile_cols(void) { return tma::TILE_COLS; }

void oracle_java_random(int64_t seed, int32_t bound, int32_t count, int32_t* out) {
    JavaRandom r(seed);
    for (int i = 0; i < count; ++i) out[i] = r.nextInt(bound);
}

}  // extern "C"
