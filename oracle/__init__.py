"""oracle/ — CPU restatement of the reference hot path.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg may
import this package.  PARITY UNPINNED (see nnet_oracle.cpp header): the reference has no
tests or golden vectors and cannot run here (no JVM).
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_RELAXED_SM = False

MODES = {"canonical": 0, "relaxed": 1, "random_n": 2, "random_nlogn": 3, "random_logn": 4}


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE])


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(_HERE, "liboracle.so")
        srcs = [os.path.join(_HERE, f) for f in ("nnet_oracle.cpp", "csw_l1.cpp")]
        srcs.append(os.path.join(os.path.dirname(_HERE), "fastneighbornet_b200", "csrc", "fnn_relaxed_sm.h"))
        srcs.append(os.path.join(os.path.dirname(_HERE), "fastneighbornet_b200", "csrc", "fnn_tile_iter.h"))
        srcs.append(os.path.join(os.path.dirname(_HERE), "fastneighbornet_b200", "csrc", "fnn_record.h"))
        if not os.path.exists(so) or any(os.path.exists(s_) and os.path.getmtime(s_) > os.path.getmtime(so) for s_ in srcs):
            build()
        L = ctypes.CDLL(so)
        c_dp = ctypes.POINTER(ctypes.c_double)
        c_ip = ctypes.POINTER(ctypes.c_int32)
        c_lp = ctypes.POINTER(ctypes.c_int64)
        L.oracle_order.argtypes = [ctypes.c_int, ctypes.c_int64, c_dp, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                   ctypes.c_int, c_ip, c_dp, ctypes.c_int64, c_lp, c_lp, ctypes.c_int, c_dp,
                                   ctypes.c_int64, c_lp]
        L.oracle_order.restype = ctypes.c_int
        L.oracle_rowsums.argtypes = [ctypes.c_int64, c_dp, c_dp]
        L.oracle_setup_d.argtypes = [ctypes.c_int64, c_ip, c_dp, c_dp]
        L.oracle_unconstrained_ls.argtypes = [ctypes.c_int64, c_dp, c_dp]
        L.oracle_atx.argtypes = [ctypes.c_int64, c_dp, c_dp]
        L.oracle_ab.argtypes = [ctypes.c_int64, c_dp, c_dp]
        c_bp = ctypes.POINTER(ctypes.c_uint8)
        L.oracle_split_weights.argtypes = [ctypes.c_int64, c_dp, c_dp, ctypes.c_int, c_lp, ctypes.c_int64, ctypes.c_int64, c_bp]
        L.oracle_l1_ab.argtypes = [ctypes.c_int64, c_dp, c_dp]
        L.oracle_l1_atx.argtypes = [ctypes.c_int64, c_dp, c_dp]
        L.oracle_l1_tree_sum.argtypes = [c_dp, ctypes.c_int64]
        L.oracle_l1_tree_sum.restype = ctypes.c_double
        L.oracle_l1_split_weights.argtypes = [ctypes.c_int64, c_dp, c_dp, c_lp, ctypes.c_int64, ctypes.c_int64, c_bp]
        L.oracle_set_relaxed_sm.argtypes = [ctypes.c_int]
        L.oracle_java_random.argtypes = [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, c_ip]
        L.oracle_tile_sequence.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_ip, c_ip, ctypes.c_int64]
        L.oracle_tile_sequence.restype = ctypes.c_int64
        _LIB = L
    return _LIB


def _dp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def _ip(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))


def _lp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))


def _bp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))


def order(D, mode="canonical", seed=12345, mult=5, additive=False, fallback=1024, want_trace=True, threads=1, max_iters=0,
          want_record=False):
    """Returns (ordering[n+1] int32, trace[k,8] float64, counters dict).  D is copied.
    max_iters = K > 0: stop after K agglomeration iterations; the trace is then the first K rows of the full trace and the
    ordering is undefined (all zeros).  0 = no limit.
    want_record: counters["record"] is the strategy record of fnn_ctx_strategy_record, one row per trace row ([k,4] int64,
    digest in column 3; view it as uint64).  Relaxed then runs through the product's state machine (set_relaxed_sm), which
    asks for the row scans in the device's order; tests/test_relaxed_sm_cpu.py holds it to the literal restatement."""
    n = D.shape[0]
    want_trace = want_trace or want_record
    Dc = np.array(D, dtype=np.float64, order="C", copy=True)
    ordering = np.zeros(n + 1, dtype=np.int32)
    max_trace = n + 8
    trace = np.zeros((max_trace, 8), dtype=np.float64)
    ntr = np.zeros(1, dtype=np.int64)
    cnt = np.zeros(2, dtype=np.int64)
    ab = np.zeros(1, dtype=np.float64)
    record = np.zeros((max_trace, 4), dtype=np.int64)
    sm_before = _RELAXED_SM
    if want_record and mode == "relaxed":
        set_relaxed_sm(True)
    try:
        rc = lib().oracle_order(MODES[mode], n, _dp(Dc), seed, mult, int(additive), fallback, _ip(ordering),
                                _dp(trace) if want_trace else None, max_trace, _lp(ntr), _lp(cnt), int(threads), _dp(ab),
                                int(max_iters), _lp(record) if want_record else None)
    finally:
        set_relaxed_sm(sm_before)
    if rc != 0:
        raise RuntimeError(f"oracle_order rc={rc}")
    out = {"pair_evals": int(cnt[0]), "npe_would_fire": int(cnt[1]), "D_final": Dc, "alg_bytes": float(ab[0])}
    if want_record:
        out["record"] = record[: int(ntr[0])]
    return ordering, trace[: int(ntr[0])], out


def rowsums(D):
    n = D.shape[0]
    Dc = np.ascontiguousarray(D, dtype=np.float64)
    out = np.zeros(n, dtype=np.float64)
    lib().oracle_rowsums(n, _dp(Dc), _dp(out))
    return out


def setup_d(ordering, d_upper):
    n = len(ordering) - 1
    o = np.ascontiguousarray(ordering, dtype=np.int32)
    du = np.ascontiguousarray(d_upper, dtype=np.float64)
    out = np.zeros(n * (n - 1) // 2, dtype=np.float64)
    lib().oracle_setup_d(n, _ip(o), _dp(du), _dp(out))
    return out


def _vec(fn, n, v):
    v = np.ascontiguousarray(v, dtype=np.float64)
    out = np.zeros_like(v)
    fn(n, _dp(v), _dp(out))
    return out


def unconstrained_ls(n, d):
    return _vec(lib().oracle_unconstrained_ls, n, d)


def atx(n, d):
    return _vec(lib().oracle_atx, n, d)


def ab(n, b):
    return _vec(lib().oracle_ab, n, b)


def _csw_result(x, st, active, with_active):
    stats = {"cg_iters": int(st[0]), "cg_calls": int(st[1]), "outer": int(st[2]), "inner": int(st[3])}
    return (x, active.astype(bool), stats) if with_active else (x, stats)


def split_weights(n, d_pos, constrained=True, max_cg_iters=0, max_cg_calls=0, with_active=False):
    """Parity-ladder level L0: CircularSplitWeights.getWeights in the reference's own operation order (nnet_oracle.cpp).
    max_cg_iters / max_cg_calls: the budget of fnn_split_weights_budget (0 = none).  Returns (x, stats), or
    (x, active, stats) with with_active=True."""
    d = np.ascontiguousarray(d_pos, dtype=np.float64)
    x = np.zeros_like(d)
    st = np.zeros(4, dtype=np.int64)
    active = np.zeros(d.shape[0], dtype=np.uint8)
    lib().oracle_split_weights(n, _dp(d), _dp(x), int(constrained), _lp(st), int(max_cg_iters), int(max_cg_calls), _bp(active))
    return _csw_result(x, st, active, with_active)


def java_random(seed, bound, count):
    out = np.zeros(count, dtype=np.int32)
    lib().oracle_java_random(seed, bound, count, _ip(out))
    return out


def tile_sequence(m, rank, world, cta, grid):
    """The tiles CTA `cta` (of `grid` per rank) of rank `rank` (of `world`) scans for m active nodes, from the PRODUCT's
    TileIter (csrc/fnn_tile_iter.h) compiled for the host: list of (first row, first column)."""
    need = lib().oracle_tile_sequence(m, rank, world, cta, grid, None, None, 0)
    r0 = np.zeros(max(1, need), dtype=np.int32)
    c0 = np.zeros(max(1, need), dtype=np.int32)
    lib().oracle_tile_sequence(m, rank, world, cta, grid, _ip(r0), _ip(c0), need)
    return [(int(a), int(b)) for a, b in zip(r0[:need], c0[:need])]


def tile_shape():
    return lib().oracle_tile_rows(), lib().oracle_tile_cols()


def l1_ab(n, b):
    return _vec(lib().oracle_l1_ab, n, b)


def l1_atx(n, d):
    return _vec(lib().oracle_l1_atx, n, d)


def l1_split_weights(n, d_pos, max_cg_iters=0, max_cg_calls=0, with_active=False):
    """Parity-ladder level L1: the GPU's formulation and reduction trees restated on the CPU (csw_l1.cpp).
    max_cg_iters / max_cg_calls: the budget of fnn_split_weights_budget (0 = none).  Returns (x, stats), or
    (x, active, stats) with with_active=True."""
    d = np.ascontiguousarray(d_pos, dtype=np.float64)
    x = np.zeros_like(d)
    st = np.zeros(4, dtype=np.int64)
    active = np.zeros(d.shape[0], dtype=np.uint8)
    lib().oracle_l1_split_weights(n, _dp(d), _dp(x), _lp(st), int(max_cg_iters), int(max_cg_calls), _bp(active))
    return _csw_result(x, st, active, with_active)


def set_relaxed_sm(on):
    """Route the oracle's Relaxed findNodes through the PRODUCT's control state machine (csrc/fnn_relaxed_sm.h), with the
    oracle's own row scans: used by tests to hold that state machine against the literal restatement on the CPU."""
    global _RELAXED_SM
    lib().oracle_set_relaxed_sm(int(bool(on)))
    _RELAXED_SM = bool(on)
