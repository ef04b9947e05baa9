"""Model of k_prune's skip rule (csrc/fnn_order.cu, DESIGN.md §4.1): a row segment is skipped only when
LB = ((c-2)*segmin - Sx(row)) - smax > T + eps, eps = 2*delta with delta the filter slack of k_scan_tma.  T can be the exact,
role-ordered Q of any pair of the segment itself, so eps must cover the rounding of LB against that Q: for every pair,
fl(Q + eps) >= LB.  The model draws max|D| on the scales of the filter-slack test (10^-3...10^3, integer multiples of
2^-1074 up to 2^-1000, the band 2^-1074...2^-1022) and makes LB as tight as it can be (segmin = the smallest entry of the
pair, smax = the column cluster's own Sx, often all entries equal), so that without eps the rule would skip the segment
that holds the minimum."""
import math

import numpy as np


def _slack(c, dmax):
    """delta of k_scan_tma / k_prune, in the kernels' operation order."""
    return 16.0 * 1.1102230246251565e-16 * (3.0 * float(c) + 2.0) * dmax + (float(c) + 2.0) * 2.0**-1074


def _scale_of(cls, rng):
    if cls == "normal":
        return float(10.0 ** rng.uniform(-3, 3))
    if cls == "sub":
        return math.ldexp(float(rng.integers(1, 2**52)), int(rng.integers(-1074, -1052)))
    if cls == "band":
        return max(float(2.0 ** rng.uniform(-1074, -1022)), 2.0**-1074)
    return math.ldexp(float(rng.integers(1, 64)), -1074)


def _exact_qs(kind, e, cm2, sr, sc):
    """Q of the pair in both role orders, as the reference rounds it (fnn_scan_tma.cuh exact1 / exact_pp)."""
    a, b, cc, d = e
    out = []
    if kind == 0:
        for t1, t2 in ((b, cc), (cc, b)):
            dpq = (((a + t1) + t2) + d) * 0.25
            out += [(cm2 * dpq - sr) - sc, (cm2 * dpq - sc) - sr]
    elif kind == 1:
        dpq = (a + b) * 0.5
        out += [(cm2 * dpq - sr) - sc, (cm2 * dpq - sc) - sr]
    else:
        out += [(cm2 * a - sr) - sc, (cm2 * a - sc) - sr]
    return out


def _case(cls, seed):
    rng = np.random.default_rng(seed)
    need_eps = 0
    for trial in range(6000):
        c = int(rng.integers(3, 200000)) if trial % 4 else int(rng.integers(3, 40))
        dmax = _scale_of(cls, rng)
        kind = trial % 3
        if trial % 2:   # all entries equal: LB equals Q in exact arithmetic
            v = float(rng.random() * dmax)
            e = (v, v, v, v)
        else:
            e = tuple(float(x) for x in rng.random(4) * dmax)
        used = e if kind == 0 else (e[:2] if kind == 1 else e[:1])
        segmin = min(used)
        sr, sc = (float(x) for x in rng.random(2) * c * dmax)
        cm2 = float(c) - 2.0
        eps = 2.0 * _slack(c, dmax)
        lb = (cm2 * segmin - sr) - sc   # k_prune: smax = this column's own Sx, the tightest case
        for q in _exact_qs(kind, e, cm2, sr, sc):
            assert not (lb > q + eps), (cls, trial, kind, c, dmax, lb, q, eps)
            need_eps += lb > q
    return need_eps


def test_prune_slack_bounds_the_rounding_of_the_lower_bound():
    need = {cls: _case(cls, seed) for cls, seed in (("normal", 11), ("sub", 12), ("band", 13), ("edge", 14))}
    # without eps the rule would skip a segment whose pair reaches T, in the normal and in the subnormal range
    assert need["normal"] > 0 and need["sub"] > 0 and need["band"] > 0, need
