"""CPU-only: the split-weight oracles (L0: the reference's operation order, oracle/nnet_oracle.cpp; L1: the device's
formulation, oracle/csw_l1.cpp) against an independent int64 restatement of the split system, and the iteration budget both
oracles share with fnn_split_weights_budget.  The GPU parity tests (test_gpu_csw_scale.py) lean on both."""
import numpy as np
import pytest

import oracle
from helpers import (circular_metric, csw_ab_exact, csw_atx_exact, csw_design_matrix, first_collapse, integer_matrix, packed_integers,
                     seeded_ordering, tree_matrix)
from fastneighbornet_b200 import synth

MATVEC_SIZES = [4, 31, 32, 33, 1024, 1448, 1449, 2370, 4097, 8000]


@pytest.mark.parametrize("n", range(4, 13))
def test_exact_reference_equals_explicit_design_matrix(n):
    A = csw_design_matrix(n)
    rng = np.random.default_rng(n)
    for v in (rng.integers(-2**20, 2**20 + 1, A.shape[0]), np.eye(A.shape[0], dtype=np.int64)[rng.integers(A.shape[0])]):
        assert (csw_ab_exact(n, v) == A @ v).all()
        assert (csw_atx_exact(n, v) == A.T @ v).all()


@pytest.mark.parametrize("n", MATVEC_SIZES)
def test_oracle_matvecs_equal_exact_reference(n):
    """Integer vectors with |v| <= 2^20: every partial sum of every summation order is exact in fp64, so L0 and L1 - two
    different orders - must both equal the int64 result exactly."""
    rng = np.random.default_rng(1000 + n)
    v = rng.integers(-2**20, 2**20 + 1, n * (n - 1) // 2)
    vf = v.astype(np.float64)
    ab, atx = csw_ab_exact(n, v).astype(np.float64), csw_atx_exact(n, v).astype(np.float64)
    assert (oracle.ab(n, vf) == ab).all()
    assert (oracle.l1_ab(n, vf) == ab).all()
    assert (oracle.atx(n, vf) == atx).all()
    assert (oracle.l1_atx(n, vf) == atx).all()
    # the unconstrained closed form inverts A: A (2 x) = 2 d holds exactly (x is a vector of halves)
    x2 = 2.0 * oracle.unconstrained_ls(n, vf)
    assert (x2 == np.round(x2)).all()
    assert (csw_ab_exact(n, x2.astype(np.int64)) == 2 * v).all()


def _int_case(n, seed, hi):
    D = integer_matrix(n, seed, hi)
    o, _, _ = oracle.order(D)
    return oracle.setup_d(o, synth.upper_triangle(D))


@pytest.mark.parametrize("hi", [3, 6])
@pytest.mark.parametrize("n", [12, 20, 40, 80])
def test_integer_inputs_rank_ties_in_the_first_collapse(n, hi):
    """Integer distances put more negatives on the 60 % cutoff than there are slots left, so the solver's tie ranking
    (k_flag_local / k_flag_blockscan / k_sel_mark_ties) runs; tree inputs have a unique cutoff."""
    fc = first_collapse(n, _int_case(n, 100 * n + hi, hi))
    assert fc["ties"] > fc["slots"] > 0, fc
    D = tree_matrix(n, 1)
    o, _, _ = oracle.order(D)
    assert first_collapse(n, oracle.setup_d(o, synth.upper_triangle(D)))["ties"] <= 1


@pytest.mark.parametrize("level", ["l0", "l1"])
def test_oracle_budget(level):
    """max_cg_iters caps every CG call at K iterations, max_cg_calls stops right after the C-th CG call; no budget and a
    budget that never binds give the unbudgeted solve."""
    solve = oracle.split_weights if level == "l0" else oracle.l1_split_weights
    n = 40
    d = _int_case(n, 43, 3)
    x, act, st = solve(n, d, with_active=True)
    x_plain, st_plain = solve(n, d)
    assert (x == x_plain).all() and st == st_plain
    assert st["cg_calls"] >= 3 and act.any()
    per_call_max = st["cg_iters"]   # no single call runs longer than all of them together
    xb, ab, sb = solve(n, d, max_cg_iters=per_call_max, max_cg_calls=st["cg_calls"] + 1, with_active=True)
    assert (xb == x).all() and (ab == act).all() and sb == st
    for calls in (1, 2, st["cg_calls"]):
        for k in (1, 5):
            xb, ab, sb = solve(n, d, max_cg_iters=k, max_cg_calls=calls, with_active=True)
            assert sb["cg_calls"] == calls and sb["cg_iters"] <= k * calls
            assert ab.any() and (xb[ab] == 0.0).all()
    # C alone: the same path as the unbudgeted solve up to the C-th call
    xb, sb = solve(n, d, max_cg_calls=st["cg_calls"])
    assert (xb == x).all() and sb["cg_iters"] == st["cg_iters"] and sb["cg_calls"] == st["cg_calls"]


def test_oracle_budget_on_a_positive_unconstrained_solution():
    """Nothing to constrain: the budget changes nothing and the active set stays empty."""
    n = 30
    cyc, w, _, du = circular_metric(n, 3)   # dyadic positive weights on every split: the closed form is exact
    d = oracle.setup_d(np.array(cyc, dtype=np.int32), du)
    assert (oracle.unconstrained_ls(n, d) > 0).all()
    for solve in (oracle.split_weights, oracle.l1_split_weights):
        x, act, st = solve(n, d, max_cg_iters=3, max_cg_calls=1, with_active=True)
        assert (x == oracle.unconstrained_ls(n, d)).all() and not act.any() and st["cg_calls"] == 0


def test_large_integer_input_ranks_ties_across_flag_scan_chunks():
    """The input class test_gpu_csw_scale.py relies on: at n = 4097 the last tie that still gets a slot in the first collapse
    lies beyond the first 1024 x 1024 entries, so its rank needs the carry of k_flag_blockscan between chunks."""
    n = 4097
    fc = first_collapse(n, oracle.setup_d(seeded_ordering(n, n), packed_integers(n, n, 4)))
    assert fc["ties"] > fc["slots"] and fc["boundary_block"] >= 1024, fc
