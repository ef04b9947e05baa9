"""Shared input builders for the parity tests (seeded; same bytes for oracle and GPU)."""
import numpy as np

from oracle import pyref

from fastneighbornet_b200 import synth


def tree_matrix(n, seed, eps=0.05):
    return synth.additive_noise_matrix(n, seed, eps)


def integer_matrix(n, seed, hi=6):
    """Small-integer distances: exact Q ties everywhere, exercises the scan-order tie-break."""
    rng = np.random.default_rng(seed)
    A = rng.integers(1, hi, size=(n, n)).astype(np.float64)
    D = np.triu(A, 1)
    return D + D.T


def random_matrix(n, seed):
    rng = np.random.default_rng(seed)
    A = rng.random((n, n))
    D = np.triu(A, 1)
    return D + D.T


def circular_metric(n, seed):
    """Strictly positive weights on ALL circular splits of a random cycle: the cycle is then the unique circular ordering
    of the metric (up to rotation / reflection) and the weights are the unique non-negative solution."""
    rng = np.random.default_rng(seed)
    cyc = [0, 1] + (rng.permutation(n - 1) + 2).tolist()
    A = np.array(pyref.live_design_matrix(n, cyc))
    w = rng.integers(1, 64, A.shape[1]).astype(np.float64) / 64.0      # dyadic: the metric is exact in fp64
    du = A @ w
    D = np.zeros((n, n))
    D[np.triu_indices(n, 1)] = du
    return cyc, w, D + D.T, du


def canon_cycle(order):
    c = list(order[1:])
    k = c.index(1)
    c = c[k:] + c[:k]
    r = [c[0]] + c[:0:-1]
    return min(c, r)


def split_dict(n, ordering, x):
    out, k, full = {}, 0, frozenset(range(1, n + 1))
    for i in range(n):
        s = set()
        for j in range(i + 1, n):
            s.add(int(ordering[j]))
            fs = frozenset(s)
            out[fs if 1 not in fs else full - fs] = x[k]
            k += 1
    return out


# ---- split-weight system over the integers (seam B2) ------------------------------------------------------------------
# Circular positions 0..n-1; split (i, j), i < j, is the set of positions {i+1, .., j}; pair (a, b), a < b.  Both index the
# same packed row-major upper triangle.  A[(a,b), (i,j)] = 1 iff the split separates a and b (exactly one of them lies in
# it), so d = A x are the split distances of weights x and A^T y the adjoint.  The two functions below restate that
# definition in int64, independently of the solver's prefix-sum formulation; tests check them against the explicit A.

def csw_design_matrix(n):
    """The explicit A (npairs x npairs, int64) straight from the definition; for small n only."""
    a, b = np.triu_indices(n, 1)   # row k of A is pair (a[k], b[k]) ...
    i, j = a, b                    # ... and column k is split (i[k], j[k]): the same packed indexing
    inside_a = (i[None, :] < a[:, None]) & (a[:, None] <= j[None, :])
    inside_b = (i[None, :] < b[:, None]) & (b[:, None] <= j[None, :])
    return (inside_a ^ inside_b).astype(np.int64)


def csw_ab_exact(n, x):
    """d = A x in int64.  d(a,b) = m(a) + m(b) - 2 M(a,b): M(a,b) (a <= b) is the weight of the splits containing both a and
    b (i < a and j >= b), m(a) = M(a,a) the weight of the splits containing a."""
    x = np.asarray(x, dtype=np.int64)
    iu = np.triu_indices(n, 1)
    X = np.zeros((n, n), dtype=np.int64)
    X[iu] = x
    below = np.zeros_like(X)
    below[1:] = np.cumsum(X, axis=0)[:-1]                   # below[a, j] = sum over i < a of X[i, j]
    del X
    M = np.cumsum(below[:, ::-1], axis=1)[:, ::-1]         # M[a, b] = sum over i < a, j >= b of X[i, j]
    del below
    m = np.diagonal(M).copy()
    return m[iu[0]] + m[iu[1]] - 2 * M[iu]


def csw_atx_exact(n, y):
    """p = A^T y in int64.  p(i,j) = sum over a in I, b not in I of Y[a,b] with I = {i+1..j} and Y the symmetric matrix of y:
    the row sums over I minus the block Y[I, I]."""
    y = np.asarray(y, dtype=np.int64)
    iu = np.triu_indices(n, 1)
    S = np.zeros((n + 1, n + 1), dtype=np.int64)            # S[p, q] = sum over a < p, b < q of Y[a, b]
    S[1:, 1:][iu] = y
    S[1:, 1:] += S[1:, 1:].T
    rows = np.concatenate([[0], np.cumsum(S[1:, 1:].sum(axis=1))])   # rows[p] = sum over a < p of the row sums
    np.cumsum(S, axis=0, out=S)
    np.cumsum(S, axis=1, out=S)
    lo, hi = iu[0] + 1, iu[1] + 1                              # I = [lo, hi)
    block = S[hi, hi] - S[lo, hi] - S[hi, lo] + S[lo, lo]
    return (rows[hi] - rows[lo]) - block


def packed_integers(n, seed, hi):
    """Packed upper triangle of small-integer distances in [1, hi) (the distribution of integer_matrix) without the n x n
    matrix: for sizes where that matrix alone is gigabytes."""
    return np.random.default_rng(seed).integers(1, hi, n * (n - 1) // 2).astype(np.float64)


def seeded_ordering(n, seed):
    """A random circular ordering in fnn_order's layout ([0] = 0, then the taxa 1..n): any permutation is a valid input of the
    split-weight solver."""
    rng = np.random.default_rng(seed)
    return np.concatenate([[0], 1 + rng.permutation(n)]).astype(np.int32)


def first_collapse(n, d_pos):
    """The first 60 % collapse of the active-set method (CircularSplitWeights.java:282-330) on the unconstrained solution:
    negatives, entries equal to the cutoff, result slots left for them, and the 1024-entry block of the last tie that
    still gets a slot (None when every tie fits, i.e. no tie ranking)."""
    import oracle
    x = oracle.unconstrained_ls(n, d_pos)
    neg = np.sort(x[x < 0.0])
    if neg.size == 0:
        return {"negatives": 0, "ties": 0, "slots": 0, "boundary_block": None}
    nkept = int(np.ceil(0.6 * neg.size))
    cutoff = neg[nkept - 1]
    ties = np.nonzero(x == cutoff)[0]
    slots = nkept - int((x < cutoff).sum())
    return {"negatives": int(neg.size), "ties": int(ties.size), "slots": slots,
            "boundary_block": int(ties[slots - 1] // 1024) if ties.size > slots else None}


# ---- the Random strategies' first iteration, in NumPy (strategy record, fnn_ctx_strategy_record) ------------------------
# At iteration 0 every node is a singleton, so NeighborNetRandom.findNodes (:130-178) reduces to i = nextInt(n), then per
# draw j = nextInt(n - 1), j = n - 1 when j == i, i = j.  The model below generates that walk from java.util.Random's
# documented LCG with NumPy only, so it shares no code with the oracle, pyref or the device (its digest uses the vectorised
# splitmix64 of the input generator, synth.py).
_JR_A, _JR_C, _JR_MASK = np.uint64(0x5DEECE66D), np.uint64(0xB), np.uint64((1 << 48) - 1)


def jr_raw(seeds, count):
    """The first `count` 31-bit values next(31) of java.util.Random(seed) for every seed: [len(seeds), count] int64.  The
    states are built by doubling: s[t + L] = A^L s[t] + c_L (mod 2^48), uint64 products wrap mod 2^64 which 2^48 divides."""
    s0 = (np.asarray(seeds, dtype=np.int64).astype(np.uint64) ^ _JR_A) & _JR_MASK
    with np.errstate(over="ignore"):
        st = ((s0 * _JR_A + _JR_C) & _JR_MASK)[:, None]
        a, c = _JR_A, _JR_C
        while st.shape[1] < count:
            st = np.concatenate([st, (st * a + c) & _JR_MASK], axis=1)
            a, c = (a * a) & _JR_MASK, (a * c + c) & _JR_MASK
    return (st[:, :count] >> np.uint64(17)).astype(np.int64)


def jr_first_try(u, bound):
    """nextInt(bound)'s first-try value for raw values u, and whether nextInt rejects u and draws again."""
    if bound & (bound - 1) == 0:
        return (bound * u) >> 31, np.zeros(u.shape, dtype=bool)
    r = u % bound
    return r, u - r + (bound - 1) >= 2 ** 31


def random_iter0_row(seed, n, total):
    """Row 0 of the strategy record of a Random mode that makes `total` draws in iteration 0: [draws, rejected, remapped,
    digest] (digest as a Python int in [0, 2^64)), and the draws' positions i, j."""
    need = total + 64
    while True:
        u = jr_raw([seed], need)[0]
        r0, rej0 = jr_first_try(u, n)
        t0 = int(np.argmin(rej0))                           # the initial i = nextInt(n) takes the first accepted value
        r, rej = jr_first_try(u[t0 + 1:], n - 1)
        acc = np.nonzero(~rej)[0]
        if acc.size >= total:
            break
        need *= 2
    acc = acc[:total]
    j = r[acc]
    rejected = np.diff(np.concatenate([[-1], acc])) > 1       # a rejected raw value comes before the accepted one
    # j == i needs j to repeat the previous j (a remapped previous j is n - 1, out of nextInt(n - 1)'s range): walk only those
    jj = j.copy()
    remapped = np.zeros(total, dtype=bool)
    first_i = int(r0[t0])
    for k in np.nonzero(j == np.concatenate([[first_i], j[:-1]]))[0]:
        if j[k] == (jj[k - 1] if k > 0 else first_i):
            jj[k] = n - 1
            remapped[k] = True
    i = np.concatenate([[first_i], jj[:-1]])
    ks = np.arange(total, dtype=np.uint64)
    with np.errstate(over="ignore"):
        terms = synth.splitmix64(synth.splitmix64(ks) ^ ((i.astype(np.uint64) << np.uint64(32)) | jj.astype(np.uint64)))
        digest = int(terms.sum(dtype=np.uint64))
    return [total, int(rejected.sum()), int(remapped.sum()), digest], i, jj


def random_first_exception(seeds, n, draws):
    """For each seed, the index of the first exceptional draw of iteration 0 (a nextInt(n - 1) rejection or a remap), or
    `draws` if none of the first `draws` is; -1 where the initial i = nextInt(n) itself rejects.  Vectorised over seeds."""
    seeds = np.asarray(seeds, dtype=np.int64)
    u = jr_raw(seeds, draws + 1)
    i0, rej_i = jr_first_try(u[:, 0], n)
    j, rej = jr_first_try(u[:, 1:], n - 1)
    prev = np.concatenate([i0[:, None], j[:, :-1]], axis=1)   # exact up to the first exception, which is all that is used
    exc = rej | (j == prev)
    first = np.where(exc.any(axis=1), np.argmax(exc, axis=1), draws)
    return np.where(rej_i, -1, first)


def hub_matrix(n, hub, seed):
    """Integer distances in which row `hub` ties exactly with all n - 1 candidates at iteration 0 (Q(hub, q) =
    (n - 2) D[hub, q] - S_hub - S_q is the same for every q) while the other rows, random integers of ~2^17, almost never
    tie.  With S_q = D[hub, q] + B_q (B: the matrix without the hub) the ties need (n - 3) D[hub, q] - B_q = K for all q:
    one sink taxon's column makes every B_q + K a multiple of n - 3, one more entry makes the sink's own row work out."""
    rng = np.random.default_rng(seed)
    rest = np.array([t for t in range(n) if t != hub])
    z = rest[-1]                                                     # the sink
    inner = rest[:-1]
    B = np.zeros((n, n), dtype=np.int64)
    U = np.triu(rng.integers(1 << 17, 1 << 18, size=(inner.size, inner.size)), 1)
    B[np.ix_(inner, inner)] = U + U.T
    K = 12345
    # make the sum of all row sums of B[inner, inner] a multiple of n - 3 (it is even; an entry moves it by 2 d)
    tot = int(B[np.ix_(inner, inner)].sum())
    d = (-tot % (n - 3)) // 2 if (-tot % (n - 3)) % 2 == 0 else ((-tot % (n - 3)) + (n - 3)) // 2
    B[inner[0], inner[1]] += d
    B[inner[1], inner[0]] += d
    R = B[inner].sum(axis=1)
    base = rng.integers(1 << 17, 1 << 18, size=inner.size)
    B[inner, z] = base + (-(R + base + K)) % (n - 3)
    B[z, inner] = B[inner, z]
    Bsum = B.sum(axis=1)
    assert ((Bsum[rest] + K) % (n - 3) == 0).all()
    D = B.copy()
    D[hub, rest] = (Bsum[rest] + K) // (n - 3)
    D[rest, hub] = D[hub, rest]
    return D.astype(np.float64)
