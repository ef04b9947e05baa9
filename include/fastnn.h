/* fastnn.h — C ABI of libfastnn.so, the B200-native Neighbor-Net hot path.
 *
 * Drop-in boundary for JacobPorter/FastNeighborNet (pure Java, no FFI of its own): the two
 * seams a maintainer re-points through JNI are
 *   B1  ordering       FastNN.java:326-361 (new NeighborNet{Canonical,Local,Random}(D, nTaxa, ...))
 *                      + FastNN.java:378/391 (int[] ordering = myNMO.runNeighborNet()),
 *                      implemented by NetMakerOriginal.java:129-162
 *   B2  split weights  FastNN.java:401-466 (live dense NNLS) / the commented call
 *                      FastNN.java:509-511 -> CircularSplitWeights.java:67,162
 * See INTEGRATION.md for the JNI stub.  Plain pointers and sizes only; no C++/torch types.
 *
 * Conventions: every entry point returns 0 on success or a negative FNN_E_* code and sets
 * fnn_last_error().  The library never writes to stdout, never throws across the ABI, and
 * has NO CPU fallback: without a CUDA device (sm_100) every compute call fails with
 * FNN_E_NODEVICE.  All arithmetic is IEEE binary64 without FMA contraction, in the
 * reference's summation order, so the circular ordering is bit-exact.
 */
#ifndef FASTNN_H
#define FASTNN_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FNN_OK 0
#define FNN_E_ARG (-1)
#define FNN_E_NODEVICE (-2)
#define FNN_E_CUDA (-3)
#define FNN_E_NOMEM (-4)
#define FNN_E_STATE (-5)
#define FNN_E_IO (-6)
#define FNN_E_UNSUPPORTED (-7)

/* Capacity limits of the Relaxed strategy (the reference's ArrayLists grow without bound): one row scan may return at most
 * 4096 exact ties of the row minimum, one findNodes call may cache at most 16 n + 65536 tie entries and 8 n + 65536
 * candidate pairs.  Beyond that (a constant matrix or thousands of duplicate taxa with n in the thousands) the ordering
 * stops with FNN_E_STATE (device-side code 11-13) instead of returning a wrong result; Canonical and Random have no such
 * limit. */

/* NetMakerOriginal.NMMode (NetMakerOriginal.java:19-21) */
enum fnn_mode {
    FNN_CANONICAL = 0,
    FNN_RELAXED = 1,
    FNN_RANDOM_N = 2,
    FNN_RANDOM_NLOGN = 3,
    FNN_RANDOM_LOGN = 4
};

/* All knobs of the reference CLI that reach the hot path (FastNN.java:136-172) plus the
 * hard-coded constants it buries (SURVEY.md §5 "config / flags"). */
typedef struct fnn_opts {
    int32_t mode;               /* -mode, enum fnn_mode; default canonical */
    int32_t mult;               /* -mult, default 5 (NeighborNetRandom.java:47); the Random modes need mult >= 1 (with no draw
                                   the reference has no pair to join), fnn_ctx_create returns FNN_E_ARG otherwise */
    int32_t additive;           /* -additive (NeighborNetLocal.java:223) */
    int32_t canonical_fallback; /* 1024: num_active <= this uses the canonical scan (NetMakerOriginal.java:361) */
    int64_t seed;               /* java.util.Random(seed) stream for Relaxed/Random (reference is unseedable) */
    int32_t device;             /* CUDA device ordinal */
    int32_t use_graph;          /* 1: replay the per-iteration kernel sequence as a CUDA graph */
    int32_t record_trace;       /* 1: keep the per-iteration (m,c,Cx,Cy,x,y,kind,best) trace on device */
    int32_t profile_every;      /* >0: time the selection kernel of every k-th iteration with CUDA events */
    int32_t reserved[6];        /* A/B switches, 0 = production: [0]=1: the selection scan reads every row segment (no
                                   lower-bound pruning, DESIGN.md §4.1); [1]=1: sum the sequential chains on one lane instead of the
                                   collapsed exact summation; [3]=1: split weights = unconstrained closed form only;
                                   [4]: split-weight solver variant (see fnn_split_weights); [5] bit 0: u.Sx chain on the
                                   critical path instead of the forked branch, bit 1: always decide the 4-candidate pick
                                   with the exact left-to-right ComputeRx sums (no certified parallel sums) */
} fnn_opts;

typedef struct fnn_ctx fnn_ctx; /* opaque: device matrix + node tables for one problem of n taxa */

typedef struct fnn_stats {
    int64_t iterations;        /* agglomeration iterations executed */
    int64_t kernel_launches;   /* CUDA kernels launched by the last run (graph nodes counted) */
    int64_t scan_launches;     /* selection-kernel launches */
    double scan_alg_bytes;     /* sum over iterations of 4*m*(m-1) - 8*pairs + 8*m (SURVEY.md §8d) */
    double prof_scan_ms;       /* profile_every>0: summed CUDA-event time of the sampled selection launches */
    double prof_scan_bytes;    /* ... and their algorithmic bytes */
    int64_t prof_scan_samples;
    double order_ms;           /* device time of the whole ordering run (CUDA events) */
    double h2d_ms;             /* device time of the host->device matrix upload, if any */
    double reserved[8];        /* [0] 4-candidate picks decided by the certified parallel ComputeRx sums, [1] picks that
                                  needed the exact left-to-right sums (NetMakerOriginal.java:413-452), [2] [3] Relaxed / Random
                                  algorithmic bytes and units, [4] matrix bytes the selection scan fetched (pruned launches:
                                  the surviving row segments; others: their algorithmic bytes), [5] row segments (a pair row
                                  counts once) that pruned launches skipped */
} fnn_stats;

void fnn_default_opts(fnn_opts* o);
const char* fnn_last_error(void);
int fnn_device_count(void);

/* ---- context API (device-resident matrix; used by bench `value` and by tests) ---------- */
int fnn_ctx_create(const fnn_opts* o, int64_t n, fnn_ctx** out);
void fnn_ctx_destroy(fnn_ctx* c);
/* upload an n*n row-major symmetric zero-diagonal host matrix (the Java double[][] D of FastNN.java:307-312).
 * Verified domain of the ordering (bit-identical to the reference's arithmetic): finite, non-negative entries, subnormal
 * values included, with max|D| small enough that 3n*max|D| stays finite.  Negative or non-finite entries are outside
 * the contract. */
int fnn_ctx_load_host(fnn_ctx* c, const double* D_rowmajor);
/* multi-GPU upload without replicating the PCIe traffic: upload only rows [row0, row0+nrows) (nrows*n doubles, row-major);
 * the host layer moves the row blocks between the ranks over NVLink (e.g. torch.distributed.broadcast on the matrix of
 * fnn_ctx_matrix_ptr), then fnn_ctx_commit_load marks the matrix loaded (zero diagonal enforced) */
int fnn_ctx_load_host_rows(fnn_ctx* c, const double* D_rows, int64_t row0, int64_t nrows);
int fnn_ctx_commit_load(fnn_ctx* c);
/* copy from a device matrix with leading dimension ld_src (elements) */
int fnn_ctx_load_device(fnn_ctx* c, const double* dD, int64_t ld_src);
/* synthesise the SURVEY §8(d) additive-tree + noise matrix in device memory from O(n) host parameters
 * (h[n-1], a[n], slot_of_taxon[n]; see fastneighbornet_b200/synth.py) */
int fnn_ctx_synth(fnn_ctx* c, const double* h, const double* a, const int64_t* slot_of_taxon, uint64_t noise_base, double eps);
/* copy the current device matrix back in the original taxon layout (only valid before fnn_ctx_order) */
int fnn_ctx_read_matrix(fnn_ctx* c, double* D_rowmajor_out);
/* run NetMakerOriginal.runNeighborNet (NetMakerOriginal.java:129): ordering_out has n+1 entries,
 * [0]=0, [1]=1, 1-based taxon ids.  The device matrix is consumed (mutated in place like the Java D). */
int fnn_ctx_order(fnn_ctx* c, int32_t* ordering_out);
/* per-iteration trace rows of 8 doubles (m, c, Cx.id, Cy.id, x.id, y.id, kind, best); returns rows written */
int64_t fnn_ctx_trace(fnn_ctx* c, double* rows_out, int64_t max_rows);
/* per-iteration strategy record, kept with the trace (opts.record_trace = 1; otherwise FNN_E_STATE): rows of 4 int64, one
 * per trace row; returns rows written.  A row is what the selection strategy did in that iteration's findNodes:
 *   Random:  draws, draws whose nextInt rejected at least once, draws remapped because j hit i or i.nbr
 *            (NeighborNetRandom.java:144-157), digest of the drawn (i, j) positions;
 *   Relaxed: row scans, tie entries they returned, -additive look-aheads, digest of the scanned rows and their ties;
 *   all zero where the strategy did not run (canonical mode, m <= canonical_fallback, the last iteration).
 * The digest (a uint64 stored as int64) is defined in csrc/fnn_record.h; a test hook for holding the strategies to a CPU
 * restatement draw for draw. */
int64_t fnn_ctx_strategy_record(fnn_ctx* c, int64_t* rows_out, int64_t max_rows);
/* Test hook of the selection scan's pruning bounds (DESIGN.md §4.1): runs the first `iters` iterations of fnn_ctx_order on
 * the loaded matrix (which it consumes) and returns the device state after them: D_out[n*n] (slot layout), the segment
 * minima segmin_out[n * S] (S = meta_out[4] segments of 256 columns per slot), the segment maxima of Sx smax_out[S] as
 * order-preserving keys (k >> 63 ? k ^ 2^63 : ~k are the double's bits; 0 = none), Sx_out[n], and meta_out[6] =
 * {m, P2, masked cluster's base slot or -1, iterations done, S, done}. */
int fnn_ctx_prune_bounds(fnn_ctx* c, int64_t iters, double* D_out, double* segmin_out, uint64_t* smax_out, double* Sx_out,
                         int64_t* meta_out);
int fnn_ctx_stats(fnn_ctx* c, fnn_stats* out);
/* device pointer + leading dimension of the internal matrix (for zero-copy producers such as torch) */
int fnn_ctx_matrix_ptr(fnn_ctx* c, double** dptr, int64_t* ld);

/* ---- multi-GPU (one process per GPU, SURVEY §8e) --------------------------------------------
 * The selection scan is sharded: rank r scans every world-th tile of the lower triangle and the per-rank
 * (Q,i,j) partial min-locs are exchanged through peer-mapped mailboxes over NVLink inside the kernels.
 * State and matrix are replicated (every rank loads the same matrix and returns the same ordering).
 * fnn_ctx_ipc_handle writes this rank's 64-byte CUDA IPC handle; the host layer all-gathers the handles
 * (torch.distributed / MPI / files) and passes the world*64 bytes, rank-ordered, to fnn_ctx_connect.
 * Every rank must call fnn_ctx_order the same number of times on a wired context (the mailbox tags carry a per-context run
 * counter).  A peer that never posts (it failed, or skipped the call) does not hang the others: after 30 s of waiting inside
 * the kernel they stop with FNN_E_STATE (device-side code 30).  A context may be destroyed as soon as its own fnn_ctx_order
 * has returned: the last exchange of a run completes on every rank before any rank can finish. */
int fnn_ctx_ipc_handle(fnn_ctx* c, void* handle_out /* 64 bytes */);
int fnn_ctx_connect(fnn_ctx* c, int32_t rank, int32_t world, const void* handles /* world * 64 bytes */);

/* ---- one-shot seams ----------------------------------------------------------------- */
/* B1: replaces `new NeighborNetX(D, n, ...).runNeighborNet()`.  Exactly one of D_rowmajor
 * (host, n*n) or phylip_path must be non-NULL.  n<=3 returns the identity ordering
 * (NetMakerOriginal.java:133-140).  The matrix must be symmetric with a zero diagonal; the verified domain is that of
 * fnn_ctx_load_host (finite, non-negative, subnormal values included, 3n*max|D| finite). */
int fnn_order(const fnn_opts* o, const double* D_rowmajor, const char* phylip_path, int64_t n, int32_t* ordering_out);
/* fnn_order keeps its last context (device buffers, tensor map, instantiated CUDA graph) for the next call with the same n
 * and options; this releases it (the JNI shim calls it from JNI_OnUnload). */
void fnn_release_cache(void);

/* initial cluster row sums only (NetMakerOriginal.initialize, :164-191) — kernel K1, exposed for parity tests */
int fnn_rowsums(const fnn_opts* o, const double* D_rowmajor, int64_t n, double* Sx_out);

/* B2: replaces the split-weight stage of FastNN.main (FastNN.java:401-466 live dense NNLS; intended call
 * FastNN.java:509-511 -> CircularSplitWeights.getWeightedSplits/getWeights, CircularSplitWeights.java:67,162)
 * with var="ols", constrained=true.  ordering: the n+1 ints of fnn_order; d_upper: the npairs = n(n-1)/2 packed
 * upper triangle in FILE order (DistancesAndNames.get(), DistancesAndNames.java:24-38,138).  x_out[npairs] uses the
 * LIVE indexing of FastNN.java:409-418: entry (i,j), i<j, row-major upper, is the split {ordering[i+1..j]}, so the
 * `x > 1e-6` filter of FastNN.java:455-466 and OutputPrinter work unchanged.  opts.reserved[3] = 1 returns the
 * unconstrained closed form only (the `useMax && maxIterations == 1` branch, CircularSplitWeights.java:166-167).
 * stats_out (optional, 5 entries): CG iterations, CG calls, outer passes, inner passes, kernel launches. */
int fnn_split_weights(const fnn_opts* o, const int32_t* ordering, const double* d_upper, int64_t n, double* x_out,
                      int64_t* stats_out);

/* B2 with the split emission of FastNN.java:455-466 folded in (SURVEY §8f N2): solves as fnn_split_weights, keeps
 * x > cutoff (the reference's optionThreshold is 1e-6) in (i,j) row-major-upper order, compacted on the device.  Entry k is
 * the split {ordering[split_i[k]+1 .. split_j[k]]} with weight[k]; the host builds BitSets for these only (the live code
 * materialises all n(n-1)/2 of them, FastNN.java:405-419).  *n_out = number kept; FNN_E_ARG if it exceeds max_out. */
int fnn_weighted_splits(const fnn_opts* o, const int32_t* ordering, const double* d_upper, int64_t n, double cutoff,
                        int32_t* split_i, int32_t* split_j, double* weight, int64_t max_out, int64_t* n_out, int64_t* stats_out);

/* Native Phylip loader (SURVEY 8f N1; host only, needs no device).  Replaces FastNN.java:270-276 (header) and
 * DistancesAndNames.java:43-132 + FastNN.java:297-312 (rows -> packed triangle -> double[n][n]) with one multi-threaded
 * pass over the mmap'ed file.  fnn_phylip_taxa: the taxon count of line 1.  fnn_read_phylip: D_rowmajor (n*n, symmetric,
 * zero diagonal); names (optional) receives n NUL-terminated names, name_stride bytes apart (truncated to fit);
 * threads 0 = all host cores.  Every value is the correctly rounded double of its token, as Double.valueOf gives. */
int fnn_phylip_taxa(const char* phylip_path, int64_t* n_out);
int fnn_read_phylip(const char* phylip_path, int64_t n, double* D_rowmajor, char* names, int64_t name_stride, int threads);

/* Streaming Nexus emission (SURVEY 8f N2; host only).  Writes what OutputPrinter.NexusWithSplitsAndDistances prints
 * (OutputPrinter.java:8-96) from the compact output of fnn_weighted_splits / fnn_network: split k is
 * {ordering[split_i[k]+1 .. split_j[k]]} with weight[k]; member lists are generated while the line is written, no
 * n(n-1)/2 BitSets (FastNN.java:405-419).  path NULL or "-" = stdout.  names NULL = t1..tn.  D_rowmajor NULL skips the
 * Distances block (an extension: at n = 20 000 that block alone is ~6 GB of text).  Numbers are formatted like
 * Double.toString (shortest round-trip digits, JDK >= 19); fnn_java_double_to_string exposes that formatter. */
int fnn_write_nexus(const char* path, int64_t n, const char* names, int64_t name_stride, const double* D_rowmajor,
                    const int32_t* ordering, const int32_t* split_i, const int32_t* split_j, const double* weight,
                    int64_t n_splits, int threads);
int fnn_java_double_to_string(double v, char* out, int64_t out_len);

/* B1 + B2 chained with the distances kept on the device (FastNN.main without -order, FastNN.java:378-466): ordering, then
 * split weights of the SAME matrix (its packed upper triangle is taken on the device before the ordering consumes it),
 * then the kept splits as in fnn_weighted_splits.  D_rowmajor: host, n*n, symmetric, zero diagonal. */
int fnn_network(const fnn_opts* o, const double* D_rowmajor, int64_t n, double cutoff, int32_t* ordering_out,
                int32_t* split_i, int32_t* split_j, double* weight, int64_t max_out, int64_t* n_out);

/* single mat-vec / stencil of the split-weight solver on a packed npairs vector, for kernel parity tests:
 * which = 0: d = A b (calculateAb, CircularSplitWeights.java:643-731); 1: p = A^T d (calculateAtx, :603-633);
 * 2: unconstrained closed form (runUnconstrainedLS, :247-271) */
int fnn_csw_matvec(const fnn_opts* o, int32_t which, const double* v, int64_t n, double* out);

/* fnn_split_weights under an iteration budget, for parity tests at sizes whose full solve takes minutes to hours (the same
 * solver, variant selection by opts.reserved[4] included; the production entry points never set a budget):
 *   max_cg_iters = K > 0: every circularConjugateGrads call (CircularSplitWeights.java:769-831) stops after at most K
 *                         iterations (kmax = min(npairs, K) instead of npairs);
 *   max_cg_calls = C > 0: the active-set method returns right after its C-th CG call, wherever that call sits in the
 *                         loop of runActiveConjugate (:359-557).
 * 0 = no budget; with both 0 the result is that of fnn_split_weights.  The CPU oracles (oracle/csw_l1.cpp L1,
 * oracle/nnet_oracle.cpp L0) take the same two parameters with the same meaning, so a truncated solve can be compared bit
 * for bit.  x_out[npairs]: the weights when the solver returned; active_out[npairs]: 1 = split held at zero by the active
 * set; stats_out (optional, 5 entries) as in fnn_split_weights. */
int fnn_split_weights_budget(const fnn_opts* o, const int32_t* ordering, const double* d_upper, int64_t n, int64_t max_cg_iters,
                             int64_t max_cg_calls, double* x_out, uint8_t* active_out, int64_t* stats_out);

/* ---- distances from a nucleotide alignment ---------------------------------------------------
 * An alignment is n taxa x L sites of codes, row-major uint8: A=0 C=1 G=2 T=3, 4 = missing.  The loader reads U as T and the
 * IUPAC ambiguity letters R Y S W K M B D H V N, plus X - ?, as missing (case-insensitive).  For a pair (i, j), with pairwise
 * deletion: v = sites where both hold a state, m = those of them where the states differ, s = transitions among the m
 * (A<->G, C<->T), q = m - s transversions; 32-bit counts, so 1 <= L <= 2^31-1.  Binary64 without FMA, in this order:
 *   FNN_DIST_P:    d = (double)m / (double)v
 *   FNN_DIST_JC69: p = m / v;  d = -0.75 * fnn_log(1.0 - p / 0.75)
 *   FNN_DIST_K2P:  P = s / v;  Q = q / v;  d = (-0.5 * fnn_log((1.0 - 2.0 * P) - Q)) - (0.25 * fnn_log(1.0 - 2.0 * Q))
 * fnn_log (csrc/fnn_log.h) is a logarithm built from IEEE + - * / alone, so the device and the CPU oracle give the same
 * bits; it is within 1 ulp of the correctly rounded log.  A result of -0.0 (m = 0) is stored as +0.0, the diagonal is +0.0
 * and D[i][j], D[j][i] are the same bits.  A pair is undefined when v = 0 or an argument of a log is <= 0 (saturation):
 *   undefined_value NaN:            the call fails with FNN_E_ARG, fnn_last_error() names the first undefined pair (i < j,
 *                                   lowest i, then lowest j) with its v, m and s; a context is left unloaded;
 *   undefined_value finite, >= 0:   every undefined entry gets that value;
 *   anything else:                  FNN_E_ARG.
 * So every matrix these calls return lies in the verified domain of the ordering (finite, non-negative, symmetric, zero
 * diagonal).  A code above 4 is FNN_E_ARG.  The computation is deterministic: ranks of a multi-GPU run that load the same
 * codes hold the same bits.  DESIGN.md §4.4. */
enum fnn_dist_model {
    FNN_DIST_P = 0,
    FNN_DIST_JC69 = 1,
    FNN_DIST_K2P = 2
};
/* Alignment loader (host only, needs no device).  The first non-blank byte picks the format: '>' (or ';') FASTA - the name is
 * the header text up to the first whitespace, sequences may wrap over any number of lines, lines may end in CRLF, lines
 * starting with ';' are skipped; a digit: sequential relaxed PHYLIP - first line `n L`, then n lines `name<whitespace>sequence`
 * whose sequence has exactly L characters once whitespace is removed (interleaved PHYLIP is rejected).  Whitespace inside
 * sequence lines is skipped.  FNN_E_IO, with a message naming the taxon or the line and column: unequal sequence lengths, an
 * empty sequence, no sequences, a sequence count that does not match the PHYLIP header, a byte that is not a code.
 * fnn_alignment_size: n and L (FASTA: L of the first record).  fnn_read_alignment: codes[n*sites]; names (optional) receives n
 * NUL-terminated names name_stride bytes apart (truncated to fit), as fnn_read_phylip; threads 0 = all host cores. */
int fnn_alignment_size(const char* path, int64_t* n_out, int64_t* sites_out);
int fnn_read_alignment(const char* path, int64_t n, int64_t sites, uint8_t* codes, char* names, int64_t name_stride, int threads);
/* Distances of the context's n taxa (codes: n*sites) computed on its device into its own matrix, then marked loaded as
 * fnn_ctx_synth does; fnn_ctx_order consumes it like any other load.  fnn_ctx_stats afterwards: h2d_ms = upload of the codes,
 * reserved[6] = packing kernel, reserved[7] = pair kernel (CUDA-event ms). */
int fnn_ctx_load_alignment(fnn_ctx* c, const uint8_t* codes, int64_t sites, int32_t model, double undefined_value);
/* Host in, host out: D_out (n*n, row-major) on device opts->device (o NULL = defaults); needs no context. */
int fnn_distances(const fnn_opts* o, const uint8_t* codes, int64_t n, int64_t sites, int32_t model, double undefined_value,
                  double* D_out);

/* left-to-right fp64 sums of nrows (<=4) rows of length len, bit-identical to `for (i) s += x[i]`
 * (the accumulation order of ComputeRx / updateClusterDistances, NetMakerOriginal.java:549-561, :530-535),
 * computed by the parallel exact-summation kernel (csrc/fnn_exact_sum.cuh) - exposed for parity tests */
int fnn_seq_sum(const fnn_opts* o, const double* rows, int32_t nrows, int64_t len, double* out);

#ifdef __cplusplus
}
#endif
#endif /* FASTNN_H */
