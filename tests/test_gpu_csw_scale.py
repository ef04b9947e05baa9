"""Seam B2 at the sizes the split-weight solver is used at, and on inputs that reach all of its code.

The solver corrects its own errors (a slightly wrong mat-vec, reduction or collapse still converges to plausible weights),
so "production path == L1 bit for bit" has to be checked where each piece of code actually runs:
  * the mat-vecs with integer vectors, where every summation order is exact, against an int64 restatement of the split
    system (tests/helpers.py) and, with float vectors, against L1 - up to n = 8000;
  * full solves on integer distances, whose first 60 % collapse has more ties at the cutoff than slots (tie ranking);
  * solves truncated by the iteration budget of fnn_split_weights_budget, against L1 under the same budget, at the sizes
    where k_cg_persistent first uses every SM, needs the third level of its reduction tree, deals several rows to a warp,
    and at its largest size; plus grid-size, relaunch and run-to-run invariance.
Boundary sizes follow from the solver's constants (read from csrc/fnn_csw.cu) and the device's SM count."""
import os
import re
from concurrent.futures import ThreadPoolExecutor
from itertools import count

import numpy as np
import pytest

import oracle
from fastneighbornet_b200 import synth
from helpers import (csw_ab_exact, csw_atx_exact, first_collapse, integer_matrix, packed_integers, seeded_ordering,
                     tree_matrix)

pytestmark = pytest.mark.gpu

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
with open(os.path.join(_ROOT, "fastneighbornet_b200", "csrc", "fnn_csw.cu")) as _f:
    _SRC = _f.read()


def _const(pattern):
    return int(re.search(pattern, _SRC).group(1))


CGP_THREADS = _const(r"constexpr int CGP_THREADS = (\d+);")     # threads per CTA of k_cg_persistent
CGP_MAX_N = _const(r"constexpr int CGP_MAX_N = (\d+);")         # largest n of the persistent path
LIT_MAX_N = _const(r"constexpr int MAX_N = (\d+);")             # largest n of the literal-order path
ENTRIES_PER_CTA = _const(r"want = \(c\.np \+ \d+\) / (\d+);")   # grid = min(SMs, ceil(npairs / ENTRIES_PER_CTA))
TREE_BLOCK = 1024                                               # values per block of the fixed reduction tree

MATVEC_SIZES = [4, 31, 32, 33, 1024, 1448, 1449, 2370, 4097, 8000]
SCALE_LABELS = ["full_grid-1", "full_grid", "level3-1", "level3", "multi_row", "4097"]
STAT_KEYS = ("cg_iters", "cg_calls", "outer", "inner")


def _npairs(n):
    return n * (n - 1) // 2


def boundary_sizes(sms):
    """n at which k_cg_persistent first runs on every SM, first needs a third level in cgp_reduce (more than 1024 level-1
    blocks), first deals more than one row to a warp in its row-scan phases, and one size past 2^12."""
    full = next(n for n in count(4) if -(-_npairs(n) // ENTRIES_PER_CTA) >= sms)
    level3 = next(n for n in count(4) if -(-_npairs(n) // TREE_BLOCK) > TREE_BLOCK)
    multi_row = sms * (CGP_THREADS // 32) + 2          # n - 1 rows > warps of the whole grid
    return {"full_grid-1": full - 1, "full_grid": full, "level3-1": level3 - 1, "level3": level3, "multi_row": multi_row,
            "4097": 4097}


def budget(n):
    """(K, C): CG iterations per call, CG calls.  The L1 oracle pays about n^2 / 4e7 s per iteration (one core)."""
    return (16, 2) if n > 4000 else (24, 3)


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _stats(st):
    return tuple(st[k] for k in STAT_KEYS)


def _same(got, want):
    """(x, active, stats) of the device against (x, active, stats) of L1: every bit and every counter."""
    x, act, st = got
    x1, a1, s1 = want
    assert _stats(st) == _stats(s1), (st, s1)
    assert (act == a1).all(), int((act != a1).sum())
    assert (x.view(np.int64) == x1.view(np.int64)).all(), (int((x != x1).sum()), float(np.abs(x - x1).max()))


# ------------------------------------------------------------------------------------------------ 1. mat-vecs
def _int_vector(n, seed):
    return np.random.default_rng(seed).integers(-2**20, 2**20 + 1, _npairs(n))


@pytest.mark.parametrize("n", MATVEC_SIZES)
def test_matvecs_exact_on_integer_vectors_and_bit_exact_vs_l1(fnn, n):
    """|v| <= 2^20: all partial sums are exact in fp64, so the device's order must give the int64 result exactly."""
    v = _int_vector(n, n)
    vf = v.astype(np.float64)
    assert (fnn.csw_matvec("ab", vf, n) == csw_ab_exact(n, v).astype(np.float64)).all()
    assert (fnn.csw_matvec("atx", vf, n) == csw_atx_exact(n, v).astype(np.float64)).all()
    x = fnn.csw_matvec("unconstrained", vf, n)
    assert (x == oracle.unconstrained_ls(n, vf)).all()
    assert (csw_ab_exact(n, (2.0 * x).astype(np.int64)) == 2 * v).all()   # the closed form inverts A exactly
    rng = np.random.default_rng(10 + n)
    for w in (rng.random(_npairs(n)), rng.normal(0.0, 1.0, _npairs(n))):
        assert (fnn.csw_matvec("ab", w, n) == oracle.l1_ab(n, w)).all()
        assert (fnn.csw_matvec("atx", w, n) == oracle.l1_atx(n, w)).all()


@pytest.mark.parametrize("n", sorted({s for s in MATVEC_SIZES if s <= LIT_MAX_N} | {LIT_MAX_N}))
def test_literal_matvecs_exact_on_integer_vectors_and_bit_exact_vs_l0(fnn, n):
    v = _int_vector(n, 7 * n)
    vf = v.astype(np.float64)
    assert (fnn.csw_matvec("ab", vf, n, variant="literal") == csw_ab_exact(n, v).astype(np.float64)).all()
    assert (fnn.csw_matvec("atx", vf, n, variant="literal") == csw_atx_exact(n, v).astype(np.float64)).all()
    w = np.random.default_rng(n).normal(0.0, 1.0, _npairs(n))
    assert (fnn.csw_matvec("ab", w, n, variant="literal") == oracle.ab(n, w)).all()
    assert (fnn.csw_matvec("atx", w, n, variant="literal") == oracle.atx(n, w)).all()


def test_literal_path_refuses_sizes_beyond_its_limit(fnn):
    n = LIT_MAX_N + 1
    with pytest.raises(fnn.FastNNError) as e:
        fnn.csw_matvec("ab", np.zeros(_npairs(n)), n, variant="literal")
    assert e.value.code == -1
    with pytest.raises(fnn.FastNNError) as e:
        fnn.split_weights_budget(seeded_ordering(n, 1), np.ones(_npairs(n)), 1, 1, variant="literal")
    assert e.value.code == -1


# ------------------------------------------------------------------------------------------------ 2. full integer solves
@pytest.fixture(scope="module")
def integer_cases():
    """(n, hi) -> ordering, packed distances, d in circular order, L1 (x, active, stats); computed once per input."""
    cache = {}

    def get(n, hi):
        if (n, hi) not in cache:
            D = integer_matrix(n, 100 * n + hi, hi)
            o, _, _ = oracle.order(D)
            du = synth.upper_triangle(D)
            d = oracle.setup_d(o, du)
            cache[(n, hi)] = (o, du, d, oracle.l1_split_weights(n, d, with_active=True))
        return cache[(n, hi)]
    return get


@pytest.mark.parametrize("variant", ["default", "graph", "literal"])
@pytest.mark.parametrize("hi", [3, 6])
@pytest.mark.parametrize("n", [12, 20, 40, 80])
def test_full_solve_on_integer_distances(fnn, integer_cases, n, hi, variant):
    """default and graph against L1, literal against L0: weights, active set and all four counters."""
    o, du, d, l1 = integer_cases(n, hi)
    fc = first_collapse(n, d)
    assert fc["ties"] > fc["slots"] > 0, fc          # the tie-ranking kernels run in the first collapse
    got = fnn.split_weights_budget(o, du, variant=variant)
    want = oracle.split_weights(n, d, with_active=True) if variant == "literal" else l1
    _same(got, want)


@pytest.mark.parametrize("variant", ["default", "graph", "literal"])
def test_no_budget_is_split_weights(fnn, integer_cases, variant):
    o, du, _, _ = integer_cases(80, 6)
    x, _, st = fnn.split_weights_budget(o, du, 0, 0, variant=variant)
    x2, st2 = fnn.split_weights(o, du, variant=variant)
    assert (x.view(np.int64) == x2.view(np.int64)).all() and st == st2


# ------------------------------------------------------------------------------------------------ 3-6. budgeted solves
class _Case:
    def __init__(self, n, kind, seed, pool):
        self.n, self.kind = n, kind
        self.o = seeded_ordering(n, seed)
        self.du = packed_integers(n, seed, 4) if kind == "int" else synth.upper_triangle(tree_matrix(n, seed))
        self.K, self.C = budget(n)
        d = oracle.setup_d(self.o, self.du)
        self.collapse = first_collapse(n, d) if kind == "int" else None
        self._l1 = pool.submit(oracle.l1_split_weights, n, d, self.K, self.C, True)

    def l1(self):
        return self._l1.result()

    def run(self, fnn, variant="default"):
        return fnn.split_weights_budget(self.o, self.du, self.K, self.C, variant=variant)


@pytest.fixture(scope="module")
def scale(sms):
    """Every budgeted input of this module, its L1 reference started at once on a thread pool (the oracle is one thread per
    solve and releases the GIL)."""
    oracle.lib()
    pool = ThreadPoolExecutor(max_workers=max(1, min(8, os.cpu_count() or 1)))
    sizes = boundary_sizes(sms)
    cases = {(label, kind): _Case(sizes[label], kind, sizes[label] + (kind == "int"), pool)
             for label in SCALE_LABELS for kind in ("tree", "int")}
    cases[("n300", "tree")] = _Case(300, "tree", 300, pool)
    yield cases
    pool.shutdown(cancel_futures=True)


@pytest.mark.parametrize("kind", ["tree", "int"])
@pytest.mark.parametrize("label", SCALE_LABELS)
def test_budgeted_solve_bit_exact_vs_l1(fnn, scale, label, kind):
    """default (k_cg_persistent) and graph (launch per phase) against L1 under the same budget: x, active set, counters.
    The kernel-launch counts show the persistent kernel actually ran."""
    c = scale[(label, kind)]
    if kind == "int":
        assert c.collapse["ties"] > c.collapse["slots"], c.collapse
    want = c.l1()
    assert want[2]["cg_calls"] == c.C
    a = c.run(fnn)
    b = c.run(fnn, "graph")
    _same(a, want)
    _same(b, want)
    assert a[2]["kernel_launches"] < b[2]["kernel_launches"] / 10


def test_some_budgeted_input_ranks_ties_across_flag_scan_chunks(scale):
    """At least one integer input's first collapse decides a tie beyond the first 1024 flag-scan blocks, where its rank
    depends on the carry k_flag_blockscan passes between chunks of 1024 blocks."""
    blocks = [c.collapse["boundary_block"] for (_, kind), c in scale.items() if kind == "int"]
    assert max(b for b in blocks if b is not None) >= TREE_BLOCK, blocks


@pytest.mark.parametrize("offset", [0, 1])
def test_largest_persistent_size_and_first_graph_only_size(fnn, offset):
    """n = CGP_MAX_N: the largest shared-memory request of k_cg_persistent (2 n doubles); n = CGP_MAX_N + 1 takes the graph
    path.  The persistent kernel must really run at CGP_MAX_N (no silent fall-back): far fewer launches than the graph path.
    The L1 oracle needs about 8 GB of host memory and half a minute here, hence K = 2 and C = 1."""
    n = CGP_MAX_N + offset
    o, du = seeded_ordering(n, n), packed_integers(n, n, 4)
    got = [fnn.split_weights_budget(o, du, 2, 1, variant=v) for v in ("default", "graph")]
    want = oracle.l1_split_weights(n, oracle.setup_d(o, du), 2, 1, with_active=True)
    for g in got:
        _same(g, want)
    la, lb = got[0][2]["kernel_launches"], got[1][2]["kernel_launches"]
    if offset == 0:
        assert la < lb / 10, (la, lb)
    else:
        assert la == lb, (la, lb)


@pytest.mark.parametrize("grid", ["1", "2", "3", "37", "sms"])
@pytest.mark.parametrize("case", [("n300", "tree"), ("level3", "int")])
def test_grid_size_does_not_change_a_bit(fnn, scale, sms, monkeypatch, case, grid):
    monkeypatch.setenv("FNN_CSW_GRID", str(sms) if grid == "sms" else grid)
    c = scale[case]
    _same(c.run(fnn), c.l1())


@pytest.mark.parametrize("per_launch", [1, 2, 7])
def test_relaunching_does_not_change_a_bit_budgeted(fnn, scale, monkeypatch, per_launch):
    """k_cg_persistent leaves after FNN_CSW_ITERS_PER_LAUNCH iterations and the next launch resumes from Scalars and the
    barrier words."""
    c = scale[("level3", "int")]
    whole = c.run(fnn)
    monkeypatch.setenv("FNN_CSW_ITERS_PER_LAUNCH", str(per_launch))
    split = c.run(fnn)
    _same(split, c.l1())
    _same(split, whole)
    st, st0 = split[2], whole[2]
    assert st["kernel_launches"] - st0["kernel_launches"] >= st["cg_iters"] / per_launch - st["cg_calls"]


@pytest.mark.parametrize("per_launch", [1, 2, 7])
def test_relaunching_does_not_change_a_bit_full_solve(fnn, integer_cases, monkeypatch, per_launch):
    o, du, _, l1 = integer_cases(80, 3)
    whole = fnn.split_weights_budget(o, du)
    monkeypatch.setenv("FNN_CSW_ITERS_PER_LAUNCH", str(per_launch))
    split = fnn.split_weights_budget(o, du)
    _same(split, l1)
    _same(split, whole)
    assert split[2]["kernel_launches"] > whole[2]["kernel_launches"]


def test_same_solve_twice_gives_the_same_bits(fnn, scale):
    c = scale[("multi_row", "int")]
    a, b = c.run(fnn), c.run(fnn)
    _same(a, b)
    assert a[2]["kernel_launches"] == b[2]["kernel_launches"]
