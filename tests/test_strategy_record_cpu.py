"""CPU-only: the per-iteration strategy record (fnn_ctx_strategy_record) of the oracle, pinned before any GPU test relies on
it.  The oracle's Random rows must equal those of the independently written Python restatement (oracle/pyref.py, its own
splitmix64), row 0 must equal a NumPy model of iteration 0 that shares no code with either, and the digest must tell
seeds and iterations apart, so that equality of two records is not vacuous.  Also: a Random mode with mult < 1 is refused
before any device is touched."""
import numpy as np
import pytest

import oracle
from oracle import pyref
from helpers import integer_matrix, random_iter0_row, random_first_exception, random_matrix, tree_matrix

RANDOM_MODES = ["random_n", "random_nlogn", "random_logn"]


def _record(D, mode, seed, fallback=4, mult=5, max_iters=0):
    _, tr, info = oracle.order(D, mode=mode, seed=seed, fallback=fallback, mult=mult, max_iters=max_iters, want_record=True)
    return tr, info["record"]


def _digests(rec):
    return rec[:, 3].copy().view(np.uint64)


def _total(mode, m, mult):
    lg = int(np.ceil(np.log10(m)))
    return {"random_n": m, "random_logn": lg, "random_nlogn": lg * m}[mode] * mult


@pytest.mark.parametrize("mode", RANDOM_MODES)
def test_oracle_record_equals_pyref(mode):
    for n in (4, 5, 6, 7, 9, 16, 31, 40):
        for seed in (1, 2):
            for D in (tree_matrix(n, seed, 0.0), tree_matrix(n, seed, 0.1), integer_matrix(n, seed), random_matrix(n, seed)):
                tr, rec = _record(D, mode, 99)
                nn = pyref.NeighborNet([list(map(float, r)) for r in D], n, mode=mode, seed=99, fallback=4)
                nn.run()
                ref = np.array(nn.record, dtype=object)
                assert rec.shape == (len(nn.trace), 4) and rec.shape[0] == tr.shape[0]
                assert (rec[:, :3] == ref[:, :3].astype(np.int64)).all(), (n, seed)
                assert _digests(rec).tolist() == [int(v) for v in ref[:, 3]], (n, seed)
                # the strategy runs while m > fallback = 4: those rows and only those are non-zero
                ran = tr[:, 0] > 4
                assert (rec[ran, 0] == [_total(mode, int(m), 5) for m in tr[ran, 0]]).all()
                assert (rec[~ran] == 0).all()


def test_record_rows_of_relaxed_count_scans():
    """Relaxed rows through the product's state machine: scans happen in every strategy iteration, every scan returns at
    least one tie, look-aheads only with -additive, and canonical iterations stay zero."""
    D = integer_matrix(40, 3)
    for additive in (False, True):
        _, tr, info = oracle.order(D, mode="relaxed", seed=7, fallback=8, additive=additive, want_record=True)
        rec = info["record"]
        ran = tr[:, 0] > 8
        assert (rec[ran, 0] >= 1).all() and (rec[ran, 1] >= rec[ran, 0]).all()
        assert (rec[~ran] == 0).all()
        assert (rec[:, 2].sum() > 0) == additive
        assert len(set(_digests(rec[ran]).tolist())) == ran.sum()


@pytest.mark.parametrize("mode", RANDOM_MODES + ["relaxed"])
def test_digests_differ_between_seeds_and_iterations(mode):
    D = tree_matrix(60, 3, 0.05)
    _, r1 = _record(D, mode, 1, fallback=8)
    _, r2 = _record(D, mode, 2, fallback=8)
    d1, d2 = _digests(r1), _digests(r2)
    ran = r1[:, 0] > 0
    assert ran.sum() > 40
    assert len(set(d1[ran].tolist())) == ran.sum()           # every iteration's digest differs
    assert (d1[ran] != d2[ran]).all()                         # and differs from the other seed's


def test_record_is_a_prefix_under_an_iteration_budget():
    D = integer_matrix(50, 4)
    for mode in RANDOM_MODES + ["relaxed"]:
        _, full = _record(D, mode, 5, fallback=8)
        for k in (1, 7, 30):
            _, pre = _record(D, mode, 5, fallback=8, max_iters=k)
            assert (pre == full[:k]).all(), (mode, k)


@pytest.mark.parametrize("mode,n,mult", [("random_n", 50, 5), ("random_nlogn", 300, 3), ("random_logn", 1000, 40),
                                         ("random_n", 1025, 2), ("random_n", 4096, 4)])
def test_numpy_model_reproduces_row_0(mode, n, mult):
    """Iteration 0 from java.util.Random's LCG in NumPy: (draws, rejections, remaps, digest) equal the oracle's row 0."""
    D = integer_matrix(n, 1)
    for seed in (3, 12345):
        _, rec = _record(D, mode, seed, fallback=8, mult=mult, max_iters=1)
        row, _, _ = random_iter0_row(seed, n, _total(mode, n, mult))
        assert rec[0, :3].tolist() == row[:3] and int(_digests(rec)[0]) == row[3]


def test_numpy_model_sees_rejections_and_remaps():
    """At n = 20 000 a nextInt(19 999) rejects about once per 10^5 draws and j hits i once per 2 * 10^4: the model's row 0 of
    a 500 000-draw Random_NLOGN iteration has both, and the oracle agrees on the whole row."""
    n = 20000
    row, i, j = random_iter0_row(777, n, _total("random_nlogn", n, 5))
    assert row[1] >= 1 and row[2] >= 10
    assert (i != j).all() and (0 <= j).all() and (j < n).all()


def test_first_exception_search():
    """The seed search of the GPU tests: draws before the first exception it reports have none, that draw has one."""
    n = 20000
    seeds = np.arange(9150, 9160)
    first = random_first_exception(seeds, n, 50)
    assert 0 in first.tolist()                                 # seed 9155: draw 0 is exceptional
    for s, f in zip(seeds.tolist(), first.tolist()):
        assert f >= 0
        before, _, _ = random_iter0_row(s, n, f)
        assert before[1] + before[2] == 0
        if f < 50:
            upto, _, _ = random_iter0_row(s, n, f + 1)
            assert upto[1] + upto[2] >= 1


@pytest.mark.parametrize("mult", [0, -1])
@pytest.mark.parametrize("mode", RANDOM_MODES)
def test_random_mult_below_one_is_refused(fnn, mode, mult):
    """With no draw the reference has no Cx (NullPointerException) and the device would select from an empty pair list: the
    context refuses such options with FNN_E_ARG before it looks for a device, so this holds on a machine without one."""
    with pytest.raises(fnn.FastNNError) as e:
        fnn.Context(16, mode=mode, mult=mult)
    assert e.value.code == -1
    D = integer_matrix(16, 1)
    with pytest.raises(fnn.FastNNError) as e:
        fnn.order(D, mode=mode, mult=mult)
    assert e.value.code == -1
