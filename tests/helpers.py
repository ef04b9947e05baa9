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
