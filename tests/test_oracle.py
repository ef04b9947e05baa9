"""CPU-only: pins the oracle as far as anything can pin it (the reference has no tests, fixtures or
golden vectors and cannot run here): published java.util.Random known answers, agreement of two
independently written restatements, restatement-independent invariants, committed golden fixtures."""
import hashlib
import json
import os

import numpy as np
import pytest

import oracle
from oracle import pyref
from helpers import canon_cycle, circular_metric, integer_matrix, random_matrix, split_dict, tree_matrix
from fastneighbornet_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))


def test_java_random_known_answers():
    # widely published sequences of java.util.Random
    assert oracle.java_random(0, 10, 5).tolist() == [0, 8, 9, 7, 5]
    assert oracle.java_random(42, 10, 5).tolist() == [0, 3, 8, 4, 0]
    r = pyref.JavaRandom(42)
    assert [r.next_int(10) for _ in range(5)] == [0, 3, 8, 4, 0]
    # power-of-two bound path and a large non-power-of-two bound agree between the restatements
    for bound in (1, 2, 64, 1000, 12345, 2**30 + 7):
        r = pyref.JavaRandom(987654321)
        assert oracle.java_random(987654321, bound, 50).tolist() == [r.next_int(bound) for _ in range(50)]


def _py(D, mode, seed, fallback):
    nn = pyref.NeighborNet([list(map(float, r)) for r in D], D.shape[0], mode=mode, seed=seed, fallback=fallback)
    return np.array(nn.run()), np.array(nn.trace, dtype=np.float64)


@pytest.mark.parametrize("mode,fb", [("canonical", 1024), ("relaxed", 4), ("random_n", 4), ("random_nlogn", 4), ("random_logn", 4)])
def test_two_restatements_agree(mode, fb):
    for n in (4, 5, 6, 7, 9, 16, 31, 60):
        for seed in (1, 2):
            for D in (tree_matrix(n, seed, 0.0), tree_matrix(n, seed, 0.1), integer_matrix(n, seed), random_matrix(n, seed)):
                o1, t1, _ = oracle.order(D, mode=mode, seed=99, fallback=fb)
                o2, t2 = _py(D, mode, 99, fb)
                assert (o1 == o2).all()
                assert t1.shape == t2.shape and (t1 == t2).all()


def test_two_restatements_agree_property():
    """Property test (hypothesis): on arbitrary small symmetric matrices - tie-heavy small integers, duplicates, wide float
    ranges - the C++ restatement and the independently written object-style Python restatement give the same ordering and
    the same per-iteration trace in every mode (with and without -additive for Relaxed)."""
    hyp = pytest.importorskip("hypothesis")
    from hypothesis import given, settings, strategies as stg

    @settings(max_examples=120, deadline=None, derandomize=True)
    @given(stg.integers(4, 13), stg.integers(0, 2 ** 31 - 1), stg.sampled_from(["canonical", "relaxed", "random_n", "random_logn", "random_nlogn"]),
           stg.sampled_from(["int3", "int9", "float", "wide", "dup"]), stg.integers(0, 1000))
    def check(n, mseed, mode, kind, seed):
        rng = np.random.default_rng(mseed)
        if kind == "int3":
            A = rng.integers(1, 4, (n, n)).astype(np.float64)
        elif kind == "int9":
            A = rng.integers(1, 10, (n, n)).astype(np.float64)
        elif kind == "float":
            A = rng.random((n, n)) + 0.01
        elif kind == "wide":
            A = (rng.random((n, n)) + 0.01) * 10.0 ** rng.integers(-3, 4, (n, n))
        else:
            base = rng.random((n, n)) + 0.01
            idx = rng.integers(0, max(2, n // 2), n)
            A = base[np.ix_(idx, idx)]
        D = np.triu(A, 1)
        D = D + D.T
        o1, t1, _ = oracle.order(D, mode=mode, seed=seed, fallback=4)
        o2, t2 = _py(D, mode, seed, 4)
        assert (o1 == o2).all()
        assert t1.shape == t2.shape and (t1 == t2).all()

    check()


def _tree_clusters(h):
    """Slot intervals [l, r] that are clades of the generator's tree (Cartesian tree of the separators)."""
    out = []

    def rec(l, r):  # slots l..r, separators h[l..r-1]
        if r - l < 1:
            return
        out.append((l, r))
        k = l + int(np.argmax(h[l:r]))
        rec(l, k)
        rec(k + 1, r)

    rec(0, len(h))
    return out


@pytest.mark.parametrize("mode,fb", [("canonical", 1024), ("relaxed", 8)])
def test_additive_tree_clades_are_contiguous(mode, fb):
    """On an exact additive tree metric every clade must be an interval of the circular order
    (canonical: always; relaxed: the mutual-row-minimum rule on cluster-averaged Q is only almost
    tree-consistent - both restatements show rare violations at n=200, so a 3 % budget is allowed)."""
    budget = 0.0 if mode == "canonical" else 0.03
    for n, seed in ((12, 1), (40, 2), (97, 3), (200, 4)):
        D = tree_matrix(n, seed, 0.0)
        h, a, pi, inv = synth.tree_params(n, seed)
        o, tr, _ = oracle.order(D, mode=mode, seed=5, fallback=fb)
        assert o[0] == 0 and o[1] == 1
        assert sorted(o[1:].tolist()) == list(range(1, n + 1))
        where = np.empty(n + 1, dtype=np.int64)
        where[o[1:]] = np.arange(n)
        clades = _tree_clusters(h)
        bad = 0
        for (l, r) in clades:
            taxa = pi[l:r + 1] + 1
            p = np.sort(where[taxa])
            gaps = np.diff(np.concatenate([p, [p[0] + n]]))
            bad += int((gaps > 1).sum() > 1)
        assert bad <= budget * len(clades), (n, seed, bad, len(clades))


def test_iteration_counts_and_kinds():
    D = tree_matrix(300, 9, 0.05)
    o, tr, info = oracle.order(D)
    assert 297 <= tr.shape[0] <= 299
    assert set(tr[:, 6].astype(int).tolist()) <= {2, 3, 4, 5}
    # clusters drop by exactly one per iteration (NetMakerOriginal.java:464-487)
    assert (np.diff(tr[:, 1]) == -1).all()
    assert info["pair_evals"] == sum(int(c) * (int(c) - 1) // 2 for c in tr[tr[:, 6] != 5][:, 1])


@pytest.mark.parametrize("mode,fb,additive", [("canonical", 1024, False), ("relaxed", 8, False), ("relaxed", 8, True),
                                              ("random_n", 8, False), ("random_nlogn", 8, False), ("random_logn", 8, False)])
def test_iteration_budget_gives_a_prefix_of_the_trace(mode, fb, additive):
    """oracle.order(max_iters=K) stops after K agglomeration iterations: its trace is the first K rows of the full trace (K
    below, at and beyond the full length), whatever the mode, the thread count or the matrix."""
    for D in (tree_matrix(60, 3, 0.05), integer_matrix(45, 4, hi=4)):
        o_full, t_full, _ = oracle.order(D, mode=mode, seed=21, fallback=fb, additive=additive)
        k_full = t_full.shape[0]
        for K in (1, 2, 7, k_full // 2, k_full - 1, k_full, k_full + 5):
            for threads in (1, 3):
                o, t, _ = oracle.order(D, mode=mode, seed=21, fallback=fb, additive=additive, threads=threads, max_iters=K)
                assert t.shape == (min(K, k_full), 8)
                assert (t == t_full[:K]).all()
                if K >= k_full:
                    assert (o == o_full).all()


def test_threaded_canonical_equals_single_thread():
    D = tree_matrix(1300, 3, 0.05)
    o1, t1, _ = oracle.order(D, threads=1)
    o4, t4, _ = oracle.order(D, threads=4)
    assert (o1 == o4).all() and (t1 == t4).all()


def test_golden_fixtures():
    with open(os.path.join(HERE, "golden", "order_golden.json")) as f:
        cases = json.load(f)
    for c in cases:
        D = tree_matrix(c["n"], c["seed"], c["eps"]) if c["kind"] == "tree" else integer_matrix(c["n"], c["seed"])
        assert hashlib.sha256(D.tobytes()).hexdigest() == c["input_sha256"], "generator drifted"
        o, tr, _ = oracle.order(D)
        if c["ordering"] is not None:
            assert o.tolist() == c["ordering"]
        assert hashlib.sha256(o.astype(np.int32).tobytes()).hexdigest() == c["ordering_sha256"]
        assert hashlib.sha256(tr.tobytes()).hexdigest() == c["trace_sha256"]


def test_golden_split_weight_fixtures():
    """tests/golden/csw_golden.json freezes both levels of the split-weight parity ladder (L0 = the reference's own
    operation order, L1 = the production formulation): weights bit for bit, CG iteration counts, kept-split counts."""
    import hashlib
    import json
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "csw_golden.json")) as f:
        cases = json.load(f)
    assert len(cases) >= 5
    for g in cases:
        D = tree_matrix(g["n"], g["seed"], g["eps"])
        o, _, _ = oracle.order(D)
        d_pos = oracle.setup_d(o, synth.upper_triangle(D))
        assert hashlib.sha256(d_pos.tobytes()).hexdigest() == g["d_pos_sha256"]
        x0, s0 = oracle.split_weights(g["n"], d_pos)
        x1, s1 = oracle.l1_split_weights(g["n"], d_pos)
        assert hashlib.sha256(x0.tobytes()).hexdigest() == g["l0_sha256"] and s0["cg_iters"] == g["l0_cg_iters"]
        assert hashlib.sha256(x1.tobytes()).hexdigest() == g["l1_sha256"] and s1["cg_iters"] == g["l1_cg_iters"]
        assert int((x0 > 1e-6).sum()) == g["l0_kept"] and int((x1 > 1e-6).sum()) == g["l1_kept"]
        if g["l0_weights"] is not None:
            assert x0.tolist() == g["l0_weights"]


def test_small_n_identity():
    for n in (1, 2, 3):
        o, _, _ = oracle.order(np.zeros((n, n)))
        assert o.tolist() == list(range(n + 1))


def test_phylip_roundtrip(tmp_path):
    D = tree_matrix(37, 2, 0.05)
    p = tmp_path / "x.phy"
    synth.write_phylip(str(p), D)
    D2, names = synth.read_phylip(str(p))
    assert (D2 == D).all() and names[0] == "t1"


# ---- split weights: the parity ladder on the CPU (L0 literal, L1 GPU-order restatement, dense NNLS) ----
def _csw_problem(n, seed, eps=0.05):
    D = tree_matrix(n, seed, eps)
    o, _, _ = oracle.order(D)
    du = synth.upper_triangle(D)
    return D, o, du, oracle.setup_d(o, du)


def test_csw_matvec_formulations_agree():
    rng = np.random.default_rng(1)
    for n in (4, 5, 9, 33, 70):
        v = rng.random(n * (n - 1) // 2)
        assert np.abs(oracle.l1_ab(n, v) - oracle.ab(n, v)).max() <= 1e-13 * v.sum()
        assert np.abs(oracle.l1_atx(n, v) - oracle.atx(n, v)).max() <= 1e-13 * v.sum()


def test_csw_l0_l1_and_dense_nnls():
    from scipy.optimize import nnls
    for n, seed in ((8, 1), (12, 2), (16, 3)):
        D, o, du, d_pos = _csw_problem(n, seed)
        x0, s0 = oracle.split_weights(n, d_pos)
        x1, s1 = oracle.l1_split_weights(n, d_pos)
        A = np.array(pyref.live_design_matrix(n, o.tolist()))
        xs, _ = nnls(A, du, maxiter=100000)
        # rotated permutation (SURVEY F4): CSW indexing == live indexing, same support, ~1e-5 agreement
        assert np.abs(x0 - xs).max() < 1e-4 and np.abs(x1 - xs).max() < 1e-4
        assert (x0 >= 0).all() and (x1 >= 0).all()


def test_csw_additive_tree_reproduces_distances():
    """eps = 0: circular split weights of a tree metric reproduce the metric: A x = d."""
    n = 20
    D, o, du, d_pos = _csw_problem(n, 7, 0.0)
    x, _ = oracle.split_weights(n, d_pos)
    assert np.abs(oracle.ab(n, x) - d_pos).max() < 1e-9


# ---- a published known answer: Neighbor-Net is consistent on circular metrics (Bryant, Moulton & Spillner 2007) ----
@pytest.mark.parametrize("n,seed", [(8, 1), (13, 2), (24, 3)])
def test_consistency_on_circular_metrics(n, seed):
    cyc, w, D, du = circular_metric(n, seed)
    o, _, _ = oracle.order(D)
    assert canon_cycle(o.tolist()) == canon_cycle(cyc)                # (a)+(b): the generating cycle is recovered
    assert canon_cycle(_py(D, "canonical", 0, 1024)[0].tolist()) == canon_cycle(cyc)
    x, _ = oracle.split_weights(n, oracle.setup_d(o, du))               # (c): and so are the generating weights
    got, want = split_dict(n, o, x), split_dict(n, cyc, w)
    assert got.keys() == want.keys()
    assert max(abs(got[k] - want[k]) for k in want) < 1e-8
