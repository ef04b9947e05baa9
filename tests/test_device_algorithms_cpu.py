"""CPU models of the non-obvious device algorithms, held to brute force on adversarial inputs.  They mirror the
kernels' logic step by step (same windows, same summaries, same checks), so the reasoning that makes the GPU results
bit-exact is exercised on every CPU run, far beyond what the GPU parity tests happen to hit:

  * the collapsed exact left-to-right summation            (csrc/fnn_exact_sum.cuh)
  * the speculative parallel java.util.Random walk          (csrc/fnn_modes.cuh: k_random_walk)
  * the slack of the selection scan's filter-then-verify    (csrc/fnn_scan_tma.cuh: delta)
  * the certificate of the 4-candidate pick                 (csrc/fnn_order.cu: k_pick)
"""
import math
import struct
from fractions import Fraction

import numpy as np
import pytest

from oracle import pyref

M52 = (1 << 52) - 1
TWO53 = float(1 << 53)


def _bits(x):
    return struct.unpack("<Q", struct.pack("<d", x))[0]


def _from_bits(b):
    return struct.unpack("<d", struct.pack("<Q", b))[0]


# ------------------------------------------------------------------ exact summation model
E_INVALID, E_IDENT = 0, -1


def _segment_summary(a, pstart, pend):
    """(e, C) of one contiguous segment, as in block_exact_seq_sum phase A2."""
    if len(a) == 0 or not np.any(a != 0.0):
        return E_IDENT, 0.0
    eps = 4.0e-11
    if not (pstart > 0.0):
        return E_INVALID, 0.0
    lo, hi = _bits(pstart * (1.0 - eps)), _bits(pend * (1.0 + eps))
    eb = lo >> 52
    if eb != (hi >> 52) or eb < 123 or eb > 1923:
        return E_INVALID, 0.0
    scale = _from_bits((2098 - eb) << 52)
    C = 0.0
    for v in a:
        x = float(v) * scale
        if math.isnan(x) or math.isinf(x):
            return E_INVALID, 0.0
        R = float(np.rint(x))
        if v < 0.0 or abs(x - R) == 0.5:
            return E_INVALID, 0.0
        C += R
    if not (C < TWO53):
        return E_INVALID, 0.0
    return int(eb), C


def _coop_apply(s, es_list, cs_list, start):
    """Longest applicable prefix of the 32 summaries from `start` (coop_apply)."""
    b = _bits(s)
    es = b >> 52
    msd = float((b & M52) | (1 << 52))
    p, acc = 0, 0.0
    for lane in range(start, 32):
        e, c = es_list[lane], cs_list[lane]
        if not (e == E_IDENT or (e > 0 and e == es)):
            break
        acc += c if e > 0 else 0.0
        if not (msd + acc < TWO53):
            break
        p += 1
        last = acc
    if p > 0 and last > 0.0:
        tot = int(msd + last)
        s = _from_bits((es << 52) | (tot & M52))
    return s, start + p


def model_exact_sum(x, threads=1024, prologue=512):
    x = np.asarray(x, dtype=np.float64)
    n = len(x)
    L = max(1, (n + threads - 1) // threads)
    segs = [x[t * L:(t + 1) * L] for t in range(threads)]
    ls = np.array([s.sum() for s in segs])                       # any order: only an estimate
    excl = np.concatenate([[0.0], np.cumsum(ls)[:-1]])
    cE, cC = [], []
    for t in range(threads):
        e, c = _segment_summary(segs[t], excl[t], excl[t] + ls[t])
        cE.append(e)
        cC.append(c)
    wE, wC = [], []
    for w in range(threads // 32):
        es, cs = cE[32 * w:32 * w + 32], cC[32 * w:32 * w + 32]
        real = [e for e in es if e > 0]
        e0 = real[0] if real else E_IDENT
        agree = all(e == E_IDENT or e == e0 for e in es)
        c = sum(cs)
        ok = agree and c < TWO53
        wE.append(e0 if ok else E_INVALID)
        wC.append(c if ok else 0.0)
    s = 0.0

    def leaf(j0, j1):
        nonlocal s
        for v in x[j0:j1]:
            s = s + float(v)

    def open_warp(w, s1):
        nonlocal s
        while s1 < 32:
            s, s1 = _coop_apply(s, cE[32 * w:32 * w + 32], cC[32 * w:32 * w + 32], s1)
            if s1 >= 32:
                break
            t = 32 * w + s1
            leaf(min(t * L, n), min(t * L + L, n))
            s1 += 1

    S0 = min(32, (prologue + L - 1) // L)
    leaf(0, min(S0 * L, n))
    open_warp(0, S0)
    s2 = 1
    while s2 < 32:
        s, s2 = _coop_apply(s, wE, wC, s2)
        if s2 >= 32:
            break
        open_warp(s2, 0)
        s2 += 1
    return s


def _seq(x):
    return float(np.cumsum(np.asarray(x, dtype=np.float64))[-1])


def test_exact_sum_model_matches_sequential():
    rng = np.random.default_rng(1)
    cases = {
        "uniform": rng.random(50000),
        "lognormal": np.exp(rng.normal(0, 3, 40000)),
        "ints": rng.integers(0, 7, 30000).astype(np.float64),
        "dyadic_ties": rng.integers(1, 2**20, 20000) * 2.0**-30 + 1.0,
        "tie_storm": np.concatenate([[2.0**52], np.full(5000, 0.5), np.full(5000, 1.5)]),
        "negatives": rng.normal(0, 1, 20000),
        "sparse_negatives": np.where(rng.random(20000) < 0.001, -1.0, 1.0) * rng.random(20000),
        "subnormals": np.concatenate([rng.random(3000) * 1e-310, rng.random(3000)]),
        "huge_range": 10.0 ** rng.uniform(-200, 200, 20000),
        "crossing_exact": np.concatenate([[1.0], np.full(4096, 2.0**-52), [1.0], np.full(5000, 2.0**-52)]),
        "zeros_then": np.concatenate([np.zeros(5000), rng.random(5000)]),
        "short": rng.random(7),
        "distance_like": 2.0 + rng.random(100003) * 3.0,
    }
    for name, x in cases.items():
        assert model_exact_sum(x) == _seq(x), name


def test_exact_sum_model_actually_collapses():
    """On distance-like data nearly everything must go through summaries (the point of the algorithm)."""
    rng = np.random.default_rng(2)
    x = 2.0 + rng.random(20000)
    L = 20
    excl = np.concatenate([[0.0], np.cumsum(x)[:-1]])
    ok = sum(_segment_summary(x[t * L:(t + 1) * L], excl[t * L], excl[t * L] + x[t * L:(t + 1) * L].sum())[0] > 0 for t in range(1000))
    assert ok >= 950


# ------------------------------------------------------------------ speculative random walk model
A_, C_, MASK = 0x5DEECE66D, 0xB, (1 << 48) - 1


def _jump(s, k):
    a, c = A_, C_
    while k:
        if k & 1:
            s = (a * s + c) & MASK
        c = (c * (a + 1)) & MASK
        a = (a * a) & MASK
        k >>= 1
    return s


def _cand(u, bound):
    return (bound * u) >> 31 if bound & (bound - 1) == 0 else u % bound


def _serial_draw(rng, i, inb, m):
    """NeighborNetRandom.java:141-158 for the current position i (inb: neighbour position or -1)."""
    if inb >= 0:
        j = rng.next_int(m - 2)
        if i == j and m - 1 == inb:
            j = m - 2
        elif i == j and m - 1 != inb:
            j = m - 1
        elif inb == j and m - 2 == i:
            j = m - 1
        elif inb == j and m - 2 != i:
            j = m - 2
    else:
        j = rng.next_int(m - 1)
        if i == j:
            j = m - 1
    return j


def model_walk(seed, nbrpos, total, window=64):
    """k_random_walk: windows of speculated draws, commit up to the first exception, replay it exactly."""
    m = len(nbrpos)
    rng = pyref.JavaRandom(seed)
    cur = rng.next_int(m)
    base = rng.s
    pairs = []
    while len(pairs) < total:
        wlen = min(window, total - len(pairs))
        # raw values (one LCG step per draw), both candidates, automaton
        raws, ca, cb = [], [], []
        for d in range(wlen):
            st = _jump(base, d + 1)
            u = st >> 17
            raws.append(u)
            ca.append(_cand(u, m - 1))
            cb.append(_cand(u, m - 2))
        state = nbrpos[cur] >= 0
        jj, exc = [], wlen
        ii = cur
        for d in range(wlen):
            bound = m - 2 if state else m - 1
            j = cb[d] if state else ca[d]
            rejected = (bound & (bound - 1)) != 0 and ((raws[d] - j + bound - 1) & 0xFFFFFFFF) >= 0x80000000
            remap = (j == ii) or (nbrpos[ii] >= 0 and j == nbrpos[ii])
            if (rejected or remap) and exc == wlen:
                exc = d
            jj.append(j)
            state = nbrpos[j] >= 0
            ii = j
        ii = cur
        for d in range(exc):
            pairs.append((ii, jj[d]))
            ii = jj[d]
        cur = ii
        base = _jump(base, exc)
        if exc < wlen:   # exact replay of the exceptional draw
            r2 = pyref.JavaRandom(0)
            r2.s = base
            j = _serial_draw(r2, cur, nbrpos[cur], m)
            pairs.append((cur, j))
            cur, base = j, r2.s
    return pairs, base


def _serial_walk(seed, nbrpos, total):
    m = len(nbrpos)
    rng = pyref.JavaRandom(seed)
    i = rng.next_int(m)
    out = []
    for _ in range(total):
        j = _serial_draw(rng, i, nbrpos[i], m)
        out.append((i, j))
        i = j
    return out, rng.s


def _structure(m, frac_paired, rng):
    nbr = [-1] * m
    idx = list(rng.permutation(m))
    k = int(frac_paired * m) // 2
    for t in range(k):
        a, b = idx[2 * t], idx[2 * t + 1]
        nbr[a], nbr[b] = int(b), int(a)
    return nbr


def test_speculative_walk_model_matches_serial():
    rng = np.random.default_rng(3)
    # small m: remaps are frequent; m-1 / m-2 powers of two: the multiply-shift path of nextInt;
    # huge m: nextInt rejections (probability ~ bound / 2^31 per draw) become frequent
    for m, total in ((7, 400), (33, 3000), (34, 3000), (257, 3000), (258, 3000), (1025, 4000), (1500000000, 3000), (2000000011, 3000)):
        for frac in (0.0, 0.5, 1.0):
            if m > 10**6:
                class Sparse(dict):   # neighbour table too large to materialise: a few paired positions
                    def __init__(self, mm):
                        super().__init__()
                        self.mm = mm
                    def __len__(self):
                        return self.mm
                    def __getitem__(self, k):
                        return dict.get(self, k, -1)
                nbr = Sparse(m)
            else:
                nbr = _structure(m, frac, rng)
            for seed in (1, 2):
                got, s1 = model_walk(seed, nbr, total)
                ref, s2 = _serial_walk(seed, nbr, total)
                assert got == ref, (m, frac, seed)
                assert s1 == s2


def test_lcg_jump_ahead():
    r = pyref.JavaRandom(123)
    s0 = r.s
    for k in (0, 1, 2, 7, 8, 1000, 8191, 123456):
        s = s0
        for _ in range(k):
            s = (s * A_ + C_) & MASK
        assert _jump(s0, k) == s


# ------------------------------------------------------------------ filter slack of the selection scan
def _rn(fr):
    return float(fr)   # Fraction -> nearest double, ties to even


def _scan_slack(c, dmax):
    """The filter slack of k_scan_tma, in the kernel's operation order (fnn_scan_tma.cuh: delta)."""
    return 16.0 * 1.1102230246251565e-16 * (3.0 * float(c) + 2.0) * dmax + (float(c) + 2.0) * 2.0**-1074


def _scale_of(cls, rng):
    """max|D| of one scale class: 'normal' 10^U(-3, 3); 'sub' an integer multiple of 2^-1074 up to 2^-1000 (subnormal and
    just above); 'band' 2^U(-1074, -1022), the subnormal range itself; 'edge' an integer multiple of 2^-1074 below 64."""
    if cls == "normal":
        return float(10.0 ** rng.uniform(-3, 3))
    if cls == "sub":
        return math.ldexp(float(rng.integers(1, 2**52)), int(rng.integers(-1074, -1052)))
    if cls == "band":
        return max(float(2.0 ** rng.uniform(-1074, -1022)), 2.0**-1074)
    return math.ldexp(float(rng.integers(1, 64)), -1074)


def test_scan_filter_slack_bounds_the_rounding_difference():
    """delta = 16 * 2^-53 * (3c + 2) * max|D| + (c + 2) * 2^-1074 must dominate |q~ - q| for every role order
    (fnn_scan_tma.cuh), for max|D| from the normal range down to a few subnormal ulps.  Below 2^-1022 a rounded product
    carries an absolute error of up to 2^-1075 that no relative term covers, and the reference's rounding of Dpq is then
    multiplied by c - 2: the second term of delta."""
    for cls in ("normal", "sub", "band", "edge"):
        _scan_slack_case(cls)


def _scan_slack_case(cls):
    rng = np.random.default_rng({"normal": 4, "sub": 5, "band": 6, "edge": 7}[cls])
    worst = 0.0
    for trial in range(4000):
        c = int(rng.integers(3, 200000)) if trial % 4 else int(rng.integers(3, 40))
        dmax = _scale_of(cls, rng)
        a, b, cc, d = (float(v) for v in rng.random(4) * dmax)
        # cluster row sums are sums of <= c cluster distances, each <= dmax
        sp, sq = (float(v) for v in rng.random(2) * c * dmax)
        cm2 = float(c) - 2.0
        delta = _scan_slack(c, dmax)
        kind = trial % 3
        exact = []
        if kind == 0:      # pair x pair: both role orders of the 4-term mean and of the subtractions
            for (t1, t2) in ((b, cc), (cc, b)):
                dpq = (((a + t1) + t2) + d) * 0.25
                exact.append((cm2 * dpq - sp) - sq)
                exact.append((cm2 * dpq - sq) - sp)
            approx = _rn(Fraction(cm2 * 0.25) * Fraction((a + b) + (cc + d)) - Fraction(sp)) - sq      # fma then subtract
        elif kind == 1:    # single x pair
            dpq = (a + b) * 0.5
            exact = [(cm2 * dpq - sp) - sq, (cm2 * dpq - sq) - sp]
            approx = _rn(Fraction(cm2 * 0.5) * Fraction(a + b) - Fraction(sp)) - sq
        else:              # single x single
            exact = [(cm2 * a - sp) - sq, (cm2 * a - sq) - sp]
            approx = _rn(Fraction(cm2) * Fraction(a) - Fraction(sp)) - sq
        for q in exact:
            worst = max(worst, abs(approx - q) / delta)
            assert abs(approx - q) <= delta, (cls, trial, kind, c, dmax, approx, q, delta)
    assert worst < 0.5, (cls, worst)   # the bound has slack to spare


# ------------------------------------------------------------------ certified 4-candidate pick model (csrc/fnn_order.cu: k_pick)
U53 = 2.0 ** -53


def _seq_sum(a):
    s = 0.0
    for v in a:
        s += float(v)
    return s


def _certificate(m, f, d, terms, present):
    """Mirror of k_pick's certificate.  terms[r] = the m weighted ComputeRx terms of chain r (r = Cx, Cx.nbr, Cy, Cy.nbr);
    the kernel sums them in SOME order (here: numpy's pairwise sum of a random permutation) and bounds the difference to
    the reference's left-to-right sum.  Returns (kstar or None, exact pick)."""
    ra, rb = (0, 1, 0, 1), (2, 2, 3, 3)
    rng = np.random.default_rng(len(terms[0]) + int(abs(f)))
    R = [float(np.sum(rng.permutation(t))) for t in terms]
    A = [float(np.sum(np.abs(t))) for t in terms]
    E = [a * ((2.0 * m + 256.0) * U53) for a in A]
    Q, e, ks = {}, {}, None
    for k in range(4):
        if not present[k]:
            continue
        t = f * d[k]
        Q[k] = (t - R[ra[k]]) - R[rb[k]]
        e[k] = 1.01 * (E[ra[k]] + E[rb[k]]) + 8.0 * U53 * (abs(t) + abs(R[ra[k]]) + abs(R[rb[k]]))
        if ks is None or Q[k] < Q[ks]:
            ks = k
    cert = all(math.isfinite(Q[k]) and math.isfinite(e[k]) for k in Q)
    cert = cert and all(k == ks or Q[ks] + e[ks] < Q[k] - e[k] for k in Q)
    # the reference: left-to-right sums, strict '<' in candidate order (NetMakerOriginal.java:428-452)
    X = [_seq_sum(t) for t in terms]
    best, kx = (f * d[0] - X[0]) - X[2], 0
    for k in (1, 2, 3):
        if present[k]:
            q = (f * d[k] - X[ra[k]]) - X[rb[k]]
            if q < best:
                best, kx = q, k
    return (ks if cert else None), kx


# binary exponents by which the certificate's model inputs are scaled: none, then down through the subnormal range, where
# products carry an absolute rounding error and the bounds themselves underflow
PICK_SHIFTS = (0, -1000, -1022, -1040, -1060, -1074)


def test_summation_order_bound_of_the_certificate():
    """|left-to-right sum - any other order| <= (2m+256) * 2^-53 * sum|a| : the E of the certificate, on adversarial inputs
    (wide magnitude ranges, alternating signs, sorted either way), scaled by 2^shift down to the subnormal range (there
    every sum whose running value stays below 2^-1022 is exact, and a bound that underflows must still hold)."""
    for shift in PICK_SHIFTS:
        _summation_order_case(shift)


def _summation_order_case(shift):
    rng = np.random.default_rng(5)
    for m in (7, 100, 3001, 20000):
        for kind in range(6):
            a = rng.random(m)
            if kind == 1:
                a = a * 10.0 ** rng.integers(-8, 8, m)
            elif kind == 2:
                a = np.sort(a * 10.0 ** rng.integers(-6, 6, m))
            elif kind == 3:
                a = np.sort(a * 10.0 ** rng.integers(-6, 6, m))[::-1]
            elif kind == 4:
                a = a * np.where(rng.random(m) < 0.5, -1.0, 1.0) * 10.0 ** rng.integers(-3, 3, m)
            elif kind == 5:
                a = np.concatenate([[1e16], rng.random(m - 1)])
            a = np.ldexp(a, shift)
            seq = _seq_sum(a)
            bound = (2.0 * m + 256.0) * U53 * float(np.sum(np.abs(a)))
            for other in (float(np.sum(a)), float(np.sum(a[::-1])), float(np.sum(rng.permutation(a))), math.fsum(a),
                          _seq_sum(a[::-1])):
                assert abs(seq - other) <= bound, (m, kind, seq, other, bound)


def test_certified_pick_never_disagrees_with_the_exact_sums():
    """Whenever the certificate accepts, the candidate it names is the one the reference's exact left-to-right sums pick;
    on exact ties and near-ties it must refuse.  Random, tie and near-tie instances, with terms and distances scaled by
    2^shift down to the subnormal range."""
    for shift in PICK_SHIFTS:
        _certified_pick_case(shift)


def _certified_pick_case(shift):
    rng = np.random.default_rng(11)
    accepted = refused = 0
    for trial in range(400):
        m = int(rng.integers(5, 4000))
        f = float(m // 2)
        mode = trial % 4
        base = rng.random((4, m)) + 0.1
        if mode == 1:      # exact ties: identical chains and distances (integer-like data)
            base = np.tile(np.round(base[0] * 4.0), (4, 1))
        elif mode == 2:    # near-ties: chains that differ in one ulp-sized term
            base = np.tile(base[0], (4, 1))
            base[1, 0] = np.nextafter(base[1, 0], 2.0)
            base[3, -1] = np.nextafter(base[3, -1], 0.0)
        w = np.where(rng.random(m) < 0.5, 1.0, 0.5)
        terms = [np.ldexp(base[r], shift) * w for r in range(4)]
        d = np.ldexp(rng.random(4) if mode in (0, 3) else np.full(4, 0.5), shift)
        present = (True, bool(rng.integers(0, 2)) or mode != 0, bool(rng.integers(0, 2)) or mode != 0, False)
        present = present[:3] + (present[1] and present[2],)
        ks, kx = _certificate(m, f, d, terms, present)
        if ks is None:
            refused += 1
        else:
            accepted += 1
            assert ks == kx, (trial, mode, ks, kx)
        if mode == 1 and sum(present) > 1:
            assert ks is None   # exact ties are never certified
    assert accepted > 100 and refused > 100, (shift, accepted, refused)
