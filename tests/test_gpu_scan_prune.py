"""Lower-bound pruning of the selection scan (k_prune, DESIGN.md §4.1).

* With pruning on and off (opts.reserved[0]) the per-iteration trace and the ordering are bit-identical to each other and
  to the CPU oracle: on inputs where most row segments are skipped, on tie-heavy inputs where the bound must keep every tied
  pair, with NaN / +inf in the padding columns, and on near-tie inputs whose distances are exact decimals (tenths, thirds):
  their Q values tie in exact arithmetic and differ by a few ulps after rounding, so the winning pair's segment has a lower
  bound within the slack eps of T - without eps k_prune skips it.
* The bookkeeping itself, read back from the device after K iterations (fnn_ctx_prune_bounds): every segment minimum is at
  most every live entry of its row segment (the row itself and its pair partner excluded), and every segment maximum of Sx
  is at least the Sx of every unmasked representative of the segment.
Pruning runs from 4 096 active nodes up, so every case starts above that size."""
import functools
import os

import numpy as np
import pytest

import oracle
from helpers import integer_matrix, tree_matrix

pytestmark = pytest.mark.gpu

THREADS = os.cpu_count() or 1


def _sym(A):
    D = np.triu(A, 1)
    return D + D.T


def _zero_taxon():
    D = tree_matrix(4300, 5, 0.05)
    D[11, :] = D[:, 11] = 0.0
    return D


def _tenths():
    D = tree_matrix(4300, 21, 0.05)
    return np.round(D / D.max() * 20.0) / 10.0


_BUILDERS = {
    "tree5000": lambda: tree_matrix(5000, 7, 0.05),
    "int4300": lambda: integer_matrix(4300, 3),
    "const4200": lambda: _sym(np.ones((4200, 4200))),
    "zero_taxon4300": _zero_taxon,
    "subnormal_tree4300": lambda: np.ldexp(tree_matrix(4300, 9, 0.05), -1060),
    "int4300_2^600": lambda: np.ldexp(integer_matrix(4300, 4).astype(np.float64), 600),
    "neartie_tenths4300": _tenths,
    "neartie_int_over_10_4300": lambda: integer_matrix(4300, 6).astype(np.float64) / 10.0,
    "neartie_int_over_3_4300": lambda: integer_matrix(4300, 8).astype(np.float64) / 3.0,
}


@functools.lru_cache(maxsize=2)
def _input(name):
    D = _BUILDERS[name]()
    D.setflags(write=False)
    return D


def _poison_padding(ctx, value):
    """Fill columns [n, ld) of the context's device matrix with `value`."""
    import torch

    ptr, ld = ctx.matrix_ptr()
    n = ctx.n
    assert ld > n, (n, ld)

    class _View:
        __cuda_array_interface__ = {"shape": (n, ld), "typestr": "<f8", "data": (ptr, False), "version": 3}

    dev = torch.device("cuda", int(ctx.opts.device))
    torch.cuda.synchronize(dev)
    torch.as_tensor(_View(), device=dev)[:, n:] = value
    torch.cuda.synchronize(dev)


def _run(fnn, D, no_prune, poison=None):
    with fnn.Context(D.shape[0], record_trace=1, no_prune=no_prune) as c:
        c.load_host(np.array(D))
        if poison is not None:
            _poison_padding(c, poison)
        o = c.order()
        return o, c.trace(), c.stats()


def _same(a, b, tag):
    (oa, ta, _), (ob, tb, _) = a, b
    assert ta.shape == tb.shape, tag
    bad = np.nonzero((ta != tb).any(axis=1))[0]
    assert bad.size == 0, f"{tag}: first diverging iteration {bad[0]}: {ta[bad[0]]} vs {tb[bad[0]]}"
    assert (oa == ob).all(), tag


@pytest.mark.parametrize("name", list(_BUILDERS))
def test_pruned_scan_equals_unpruned_and_oracle(fnn, name):
    D = _input(name)
    on = _run(fnn, D, 0)
    off = _run(fnn, D, 1)
    _same(on, off, f"{name}: pruning on vs off")
    o_ref, tr_ref, _ = oracle.order(np.array(D), mode="canonical", threads=THREADS)
    _same(on, (o_ref, tr_ref, None), f"{name}: pruned vs oracle")
    assert off[2]["scan_units_skipped"] == 0
    if name.startswith("const"):   # every pair ties: the bound must keep every segment
        assert on[2]["scan_units_skipped"] == 0, on[2]
    if name.startswith("tree"):
        assert on[2]["scan_units_skipped"] > 0, name
        assert on[2]["scan_read_bytes"] < 0.5 * off[2]["scan_read_bytes"], (on[2], off[2])


@pytest.mark.parametrize("poison", [float("nan"), float("inf"), -1e308])
def test_poisoned_padding(fnn, poison):
    """n = 4 301 (ld = 4 304): the padding columns hold NaN / +inf / -1e308; no bound may read them."""
    D = tree_matrix(4301, 13, 0.05)
    on = _run(fnn, D, 0, poison)
    assert on[2]["scan_units_skipped"] > 0
    o_ref, tr_ref, _ = oracle.order(D, mode="canonical", threads=THREADS)
    _same(on, (o_ref, tr_ref, None), f"poison {poison}")


def _check_bounds(s):
    m, P2, msk = s["m"], s["P2"], s["mask_su"]
    nseg = (m + 255) // 256
    D = np.full((m, nseg * 256), np.inf)
    D[:, :m] = s["D"][:m, :m]
    idx = np.arange(m)
    D[idx, idx] = np.inf
    pr = idx[idx < P2]
    D[pr, pr ^ 1] = np.inf
    true_min = D.reshape(m, nseg, 256).min(axis=2)
    seg = s["segmin"][:m, :nseg]
    bad = np.argwhere(~(seg <= true_min))
    assert bad.size == 0, f"segmin above a live entry at (row, segment) {bad[:5].tolist()}: {seg[tuple(bad[0])]} > {true_min[tuple(bad[0])]}"
    assert np.isfinite(seg).mean() > 0.9   # the bounds are real, not a vacuous -inf
    reps = idx[((idx >= P2) | (idx % 2 == 0)) & ((idx & ~1) != msk)]
    smax = s["smax"][reps // 256]
    worse = reps[~(smax >= s["Sx"][reps])]
    assert worse.size == 0, f"smax below Sx of representatives {worse[:5].tolist()}"


@pytest.mark.parametrize("name,iters", [("tree5000", 1), ("tree5000", 400), ("tree5000", 950), ("int4300", 300),
                                        ("neartie_tenths4300", 250)])
def test_bounds_hold_against_the_device_matrix(fnn, name, iters):
    with fnn.Context(_input(name).shape[0]) as c:
        c.load_host(np.array(_input(name)))
        s = c.prune_bounds(iters)
    assert s["iter"] == iters and not s["done"]
    _check_bounds(s)


def test_bounds_hold_with_poisoned_padding(fnn):
    D = tree_matrix(4301, 13, 0.05)
    with fnn.Context(4301) as c:
        c.load_host(D)
        _poison_padding(c, float("nan"))
        s = c.prune_bounds(200)
    _check_bounds(s)


def test_prefix_at_production_size(fnn):
    """The first 56 iterations at n = 20 000 (the bench workload's generator) against the budgeted oracle, pruning on; most
    row segments are skipped."""
    from fastneighbornet_b200 import synth
    n, K = 20000, 48
    D = synth.additive_noise_matrix(n, 1, 0.05)
    with fnn.Context(n, record_trace=1) as c:
        c.load_host(D)
        c.order()
        tr = c.trace()[: K + 8]
        st = c.stats()
    _, tr_ref, _ = oracle.order(D, mode="canonical", threads=THREADS, max_iters=K + 8)
    bad = np.nonzero((tr != tr_ref[: len(tr)]).any(axis=1))[0]
    assert bad.size == 0, f"first diverging iteration {bad[0]}"
    assert st["scan_units_skipped"] > 0
