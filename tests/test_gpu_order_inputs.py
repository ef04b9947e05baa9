"""The ordering engine (seam B1) against the CPU oracle on inputs the other parity tests do not reach: copies scaled by
powers of two down to the subnormal range and up to 2^900, tie-heavy and degenerate matrices (small integers, duplicate
taxa, Phylip-rounded decimals, twelve decades of magnitude, the zero matrix, a taxon at distance 0 from all others),
sizes whose leading dimension has no padding (n % 16 == 0, the TMA boxes then run off the tensor edge) or just exceeds a
tile boundary, padding columns filled with NaN / -1e308 / +inf, and the size from which k_chain reads the u.Sx chain
from global memory instead of staging it in shared memory.  Every case compares the per-iteration trace (all 8 columns)
and the ordering with the oracle bit for bit."""
import math
import os

import numpy as np
import pytest

import oracle
from helpers import integer_matrix, tree_matrix

pytestmark = pytest.mark.gpu

THREADS = os.cpu_count() or 1
SCALES = (-1074, -1060, -1040, -1022, -600, 600, 900)
MODES = ("canonical", "relaxed", "random_n", "random_nlogn", "random_logn")


def _gpu(fnn, D, mode="canonical", seed=777, fallback=1024, additive=False, poison=None, record_trace=1):
    n = D.shape[0]
    with fnn.Context(n, record_trace=record_trace, mode=mode, seed=seed, canonical_fallback=fallback,
                     additive=int(additive)) as c:
        c.load_host(D)
        if poison is not None:
            _poison_padding(c, poison)
        o = c.order()
        return o, (c.trace() if record_trace else None)


def _check(fnn, D, mode="canonical", seed=777, fallback=1024, additive=False, what=""):
    o_ref, tr_ref, _ = oracle.order(D, mode=mode, seed=seed, fallback=fallback, additive=additive, threads=THREADS)
    o, tr = _gpu(fnn, D, mode, seed, fallback, additive)
    tag = f"{what} n={D.shape[0]} mode={mode} additive={additive}"
    assert tr.shape == tr_ref.shape, (tag, tr.shape, tr_ref.shape)
    bad = np.nonzero((tr != tr_ref).any(axis=1))[0]
    assert bad.size == 0, f"{tag}: first diverging iteration {bad[0]}: gpu={tr[bad[0]]} ref={tr_ref[bad[0]]}"
    assert (o == o_ref).all(), tag
    return o


def _sym(A):
    D = np.triu(A, 1)
    return D + D.T


# ------------------------------------------------------------------ copies scaled by 2^k
@pytest.mark.parametrize("n,mode,fallback", [(12, "canonical", 1024), (100, "canonical", 1024), (777, "canonical", 1024),
                                             (120, "relaxed", 8), (120, "random_n", 8), (120, "random_nlogn", 8)])
@pytest.mark.parametrize("kind", ["tree", "int"])
def test_scaled_copies(fnn, n, mode, fallback, kind):
    """ldexp(D, k) from 2^-1074 (every distance a handful of subnormal ulps, ties everywhere) to 2^900.  Where the oracle
    orders the scaled copy as it orders D, the GPU ordering must be scale-invariant too."""
    D = tree_matrix(n, 3, 0.05) if kind == "tree" else integer_matrix(n, 3)
    o_ref0, _, _ = oracle.order(D, mode=mode, seed=31, fallback=fallback, want_trace=False, threads=THREADS)
    o0, _ = _gpu(fnn, D, mode, 31, fallback, record_trace=0)
    assert (o0 == o_ref0).all()
    for k in SCALES:
        Dk = np.ldexp(D, k)
        assert np.isfinite(3.0 * n * Dk.max())
        o = _check(fnn, Dk, mode, 31, fallback, what=f"{kind} * 2^{k}")
        if (o == o_ref0).all():
            assert (o == o0).all()


# ------------------------------------------------------------------ input classes
def _matrix(cls, n, rng):
    """The generators of tests/test_oracle.py::test_two_restatements_agree_property, and further degenerate inputs."""
    if cls == "int3":
        return _sym(rng.integers(1, 4, (n, n)).astype(np.float64))
    if cls == "int9":
        return _sym(rng.integers(1, 10, (n, n)).astype(np.float64))
    if cls == "float":
        return _sym(rng.random((n, n)) + 0.01)
    if cls == "wide":
        return _sym((rng.random((n, n)) + 0.01) * 10.0 ** rng.integers(-3, 4, (n, n)))
    if cls == "dup":
        base = rng.random((n, n)) + 0.01
        idx = rng.integers(0, max(2, n // 2), n)
        return _sym(base[np.ix_(idx, idx)])
    if cls == "round3":   # distances as Phylip text carries them: few decimals, many exact ties
        return _sym(np.round((rng.random((n, n)) + 0.01) * 10.0, 3))
    if cls == "round5":
        return _sym(np.round(rng.random((n, n)) + 0.01, 5))
    if cls == "decades":
        return _sym((rng.random((n, n)) + 0.01) * 10.0 ** rng.uniform(-6, 6, (n, n)))
    if cls == "zero":
        return np.zeros((n, n))
    if cls == "hub":      # one taxon at distance 0 from every other
        D = _sym(rng.random((n, n)) + 0.01)
        h = int(rng.integers(0, n))
        D[h, :] = 0.0
        D[:, h] = 0.0
        return D
    raise ValueError(cls)


CLASSES = ("int3", "int9", "float", "wide", "dup", "round3", "round5", "decades", "zero", "hub")


@pytest.mark.parametrize("cls", CLASSES)
def test_input_classes_small_every_mode(fnn, cls):
    """n = 4 ... 13, every mode (Relaxed with and without -additive), canonical fallback 4: the strategies themselves run
    down to four active nodes."""
    rng = np.random.default_rng(CLASSES.index(cls) + 100)
    for n in range(4, 14):
        for rep in range(2):
            D = _matrix(cls, n, rng)
            seed = int(rng.integers(0, 1000))
            for mode in MODES:
                _check(fnn, D, mode, seed, 4, what=f"{cls} rep {rep}")
            _check(fnn, D, "relaxed", seed, 4, additive=True, what=f"{cls} rep {rep}")


@pytest.mark.parametrize("n", [300, 1300])
@pytest.mark.parametrize("cls", CLASSES)
def test_input_classes_canonical(fnn, cls, n):
    _check(fnn, _matrix(cls, n, np.random.default_rng(n + CLASSES.index(cls))), what=cls)


# ------------------------------------------------------------------ unpadded and boundary sizes
@pytest.mark.parametrize("n", [512, 1024, 2048, 4096, 513, 1025, 4097])
@pytest.mark.parametrize("kind", ["tree", "int"])
def test_unpadded_and_boundary_sizes(fnn, n, kind):
    """n % 16 == 0: the leading dimension is n, so the 256-column TMA boxes that cross column n read the tensor map's
    out-of-bounds fill, not padding; the multiples of 512 (TILE_COLS) also end exactly on a tile.  n = 513, 1025, 4097:
    one column past such a boundary."""
    D = tree_matrix(n, 5, 0.05) if kind == "tree" else integer_matrix(n, 5, hi=4)
    _check(fnn, D, what=kind)


# ------------------------------------------------------------------ poisoned padding columns
def _poison_padding(ctx, value):
    """Fill columns [n, ld) of the context's device matrix with `value` (through its __cuda_array_interface__)."""
    import torch

    ptr, ld = ctx.matrix_ptr()
    n = ctx.n
    assert ld > n, (n, ld)

    class _View:
        __cuda_array_interface__ = {"shape": (n, ld), "typestr": "<f8", "data": (ptr, False), "version": 3}

    dev = torch.device("cuda", int(ctx.opts.device))
    torch.cuda.synchronize(dev)
    view = torch.as_tensor(_View(), device=dev)
    view[:, n:] = value
    torch.cuda.synchronize(dev)
    assert bool(torch.isnan(view[:, n:]).all()) if math.isnan(value) else bool((view[:, n:] == value).all())


@pytest.mark.parametrize("n,mode", [(513, "canonical"), (1000, "canonical"), (1500, "canonical"), (4097, "canonical"),
                                    (1500, "relaxed")])
def test_poisoned_padding_columns_are_never_read(fnn, n, mode):
    """When n % 16 != 0 the columns [n, ld) are padding that nothing writes; a kernel that read them would see whatever
    the allocation held (usually zeros).  Filled with NaN, -1e308 or +inf, the trace must still be the oracle's."""
    D = tree_matrix(n, 6, 0.05)
    o_ref, tr_ref, _ = oracle.order(D, mode=mode, seed=123, threads=THREADS)
    for value in (float("nan"), -1e308, float("inf")):
        o, tr = _gpu(fnn, D, mode, 123, 1024, poison=value)
        assert tr.shape == tr_ref.shape, (value, tr.shape, tr_ref.shape)
        bad = np.nonzero((tr != tr_ref).any(axis=1))[0]
        assert bad.size == 0, f"padding={value}: first diverging iteration {bad[0]}: gpu={tr[bad[0]]} ref={tr_ref[bad[0]]}"
        assert (o == o_ref).all(), value


# ------------------------------------------------------------------ u.Sx chain read from global memory
# k_chain stages the u.Sx chain in shared memory when CHAIN_SMEM_BASE + 8 * rxs_ld <= CHAIN_SMEM_MAX, with
# CHAIN_SMEM_BASE = sizeof(xsum::SmemN<1>) = 18 056 B, CHAIN_SMEM_MAX = 220 KiB = 225 280 B and rxs_ld = n rounded up to a
# multiple of 1024 (xsum::THREADS): rxs_ld <= 25 903, i.e. n <= 25 600.  From n = 25 601 on (rxs_ld = 26 624) it reads the
# chain from global memory (csrc/fnn_order.cu, fnn_ctx_create and k_chain).
CHAIN_K = 128


@pytest.fixture(scope="module")
def chain_matrix():
    return tree_matrix(25601, 8, 0.05)


@pytest.mark.parametrize("mode", ["canonical", "relaxed"])
@pytest.mark.parametrize("n", [25600, 25601])
def test_chain_unstaged_prefix(fnn, chain_matrix, n, mode):
    """n = 25 601 (chain in global memory) and n = 25 600 (staged, the control; the leading block of the same matrix):
    the full GPU ordering with a trace, whose first 128 rows must equal the budgeted oracle; the ordering is a permutation
    and equals that of a second run without a trace (the production path: certified picks, chain on the forked branch)."""
    D = chain_matrix if n == chain_matrix.shape[0] else np.ascontiguousarray(chain_matrix[:n, :n])
    _, tr_ref, info = oracle.order(D, mode=mode, seed=2718, threads=THREADS, max_iters=CHAIN_K)
    del info
    assert tr_ref.shape == (CHAIN_K, 8)
    o, tr = _gpu(fnn, D, mode, 2718, 1024)
    assert tr.shape[0] > CHAIN_K
    bad = np.nonzero((tr[:CHAIN_K] != tr_ref).any(axis=1))[0]
    assert bad.size == 0, f"n={n} {mode}: first diverging iteration {bad[0]}: gpu={tr[bad[0]]} ref={tr_ref[bad[0]]}"
    assert o[0] == 0 and o[1] == 1 and sorted(o[1:].tolist()) == list(range(1, n + 1))
    o2, _ = _gpu(fnn, D, mode, 2718, 1024, record_trace=0)
    assert (o2 == o).all()
