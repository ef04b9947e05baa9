"""CPU-only: the split-matching rule of fnn_bootstrap (csrc/fnn_boot.cu, DESIGN.md §4.5) restated in NumPy against a
brute-force comparison of bipartitions, the Nexus writer's confidence column, and the CLI's -bootstrap checks."""
import collections
import ctypes

import numpy as np
import pytest

import fastneighbornet_b200 as fnn
from fastneighbornet_b200.__main__ import parse_args


def _row_start(n, i):
    return i * (2 * n - i - 1) // 2


def _packed(n, i, j):
    return _row_start(n, i) + (j - i - 1)


def _sparse_table(vals, op):
    levels = [np.asarray(vals)]
    k = 1
    while (1 << k) <= len(vals):
        prev, half = levels[-1], 1 << (k - 1)
        levels.append(op(prev[:len(vals) - (1 << k) + 1], prev[half:half + len(vals) - (1 << k) + 1]))
        k += 1
    return levels


def _query(levels, op, l, r):
    k = int(r - l + 1).bit_length() - 1
    return op(levels[k][l], levels[k][r - (1 << k) + 1])


def matching_rule(O, orig_kept_idx, O_r, rep_kept_idx):
    """support increments of one replicate by the device's rule: sparse tables of pos(O_r[p + 1]), the side U without
    O[n] (a complement when max pos(T) = n), contiguity of pos(U), binary search of (lo - 1, hi) in the original indices."""
    n = len(O) - 1
    pos = np.zeros(n + 1, dtype=np.int64)
    pos[O[1:]] = np.arange(1, n + 1)
    vals = pos[np.asarray(O_r[1:])]
    tmin, tmax = _sparse_table(vals, np.minimum), _sparse_table(vals, np.maximum)
    orig = np.asarray(orig_kept_idx, dtype=np.int64)
    out = np.zeros(len(orig), dtype=np.int64)
    for idx in (int(v) for v in rep_kept_idx):
        a = next(i for i in range(n - 1) if _row_start(n, i + 1) > idx)
        b = idx - _row_start(n, a) + a + 1
        lo, hi, size = int(_query(tmin, np.minimum, a, b - 1)), int(_query(tmax, np.maximum, a, b - 1)), b - a
        if hi == n:
            size = n - size
            lo, hi = int(_query(tmin, np.minimum, b, n - 1)), int(_query(tmax, np.maximum, b, n - 1))
            if a > 0:
                lo, hi = min(lo, int(_query(tmin, np.minimum, 0, a - 1))), max(hi, int(_query(tmax, np.maximum, 0, a - 1)))
        if hi - lo + 1 != size:
            continue
        k = np.searchsorted(orig, _packed(n, lo - 1, hi))
        if k < len(orig) and orig[k] == _packed(n, lo - 1, hi):
            out[k] += 1
    return out


def brute_force(O, orig_kept_idx, O_r, rep_kept_idx):
    """support increments by comparing bitsets: split k is matched when a replicate split equals it or its complement
    (both normalised to the side without taxon 1)."""
    n = len(O) - 1
    rs = np.array([_row_start(n, i) for i in range(n)], dtype=np.int64)

    def keys(order, idx):
        idx = np.asarray(idx, dtype=np.int64)
        ii = np.searchsorted(rs, idx, side="right") - 1
        jj = idx - rs[ii] + ii + 1
        out = []
        for i, j in zip(ii, jj):
            m = np.zeros(n + 1, dtype=bool)
            m[np.asarray(order[i + 1: j + 1])] = True
            m = m[1:]
            out.append((~m if m[0] else m).tobytes())
        return out

    rep = collections.Counter(keys(O_r, rep_kept_idx))
    return np.array([rep.get(k, 0) for k in keys(O, orig_kept_idx)], dtype=np.int64)


def _perturbed(O, rng, kind):
    n = len(O) - 1
    t = list(O[1:])
    if kind == "same":
        pass
    elif kind == "rotate":          # the same circle, cut elsewhere: every split comes back, many as complements
        r = int(rng.integers(1, n))
        t = t[r:] + t[:r]
    elif kind == "reverse":
        r = int(rng.integers(0, n))
        t = (t[r:] + t[:r])[::-1]
    elif kind == "swaps":
        for _ in range(int(rng.integers(1, 4))):
            a, b = rng.integers(0, n, 2)
            t[a], t[b] = t[b], t[a]
    else:
        t = list(rng.permutation(t))
    return np.array([0] + t, dtype=np.int64)


@pytest.mark.parametrize("n", [4, 5, 6, 7, 9, 16, 33, 64, 65, 130, 200])
def test_matching_rule_equals_brute_force(n):
    rng = np.random.default_rng(n)
    npairs = n * (n - 1) // 2
    trivial = [_packed(n, i, i + 1) for i in range(n - 1)] + [_packed(n, 0, n - 1)]   # singletons and the complement of {O[n]}
    with_last = [_packed(n, i, n - 1) for i in range(n - 1)]                           # splits that contain O[n] on the replicate side
    hits = 0
    for trial, kind in enumerate(["same", "rotate", "reverse", "swaps", "random"] * 2):
        O = np.array([0] + list(rng.permutation(np.arange(1, n + 1))), dtype=np.int64)
        O_r = _perturbed(O, rng, kind)
        take = min(npairs, 3 * n)
        orig = np.unique(np.concatenate([rng.choice(npairs, take, replace=False), trivial[: n // 2]]))
        rep = np.unique(np.concatenate([rng.choice(npairs, take, replace=False), trivial, with_last]))
        if trial % 2:
            orig = np.arange(npairs)   # every split of O: whatever the replicate keeps that is circular in O must be found
        got = matching_rule(O, orig, O_r, rep)
        ref = brute_force(O, orig, O_r, rep)
        assert (got == ref).all(), (n, kind)
        assert got.max(initial=0) <= 1   # distinct replicate splits are distinct bipartitions
        hits += int(got.sum())
    assert hits > 0


def _nexus_text(tmp_path, name, **kw):
    p = tmp_path / name
    fnn.write_nexus(str(p), **kw)
    return p.read_text()


def test_nexus_support_line_format(tmp_path):
    n = 9
    rng = np.random.default_rng(3)
    ordering = np.array([0] + list(rng.permutation(np.arange(1, n + 1))), dtype=np.int32)
    si = np.array([0, 0, 1, 2, 3, 5, 0], dtype=np.int32)
    sj = np.array([1, 4, 3, 8, 5, 7, 8], dtype=np.int32)
    w = np.array([0.5, 1e-3, 2.25, 7e-7, 0.125, 3.0, 1.0 / 3.0])
    R = 7
    sup = np.array([0, 7, 3, 1, 6, 2, 5], dtype=np.int32)
    plain = _nexus_text(tmp_path, "a.nex", ordering=ordering, split_i=si, split_j=sj, weight=w)
    withs = _nexus_text(tmp_path, "b.nex", ordering=ordering, split_i=si, split_j=sj, weight=w, support=sup, replicates=R)
    assert "confidences=no" in plain and "confidences=yes" not in plain
    lines = withs.split("\n")
    start = lines.index("MATRIX", lines.index("BEGIN Splits;"))
    for k in range(len(w)):
        members = " ".join(str(t) for t in sorted(int(x) for x in ordering[si[k] + 1: sj[k] + 1]))
        card = int(sj[k] - si[k])
        conf = fnn.java_double_str((100.0 * int(sup[k])) / R)
        assert lines[start + 1 + k] == f"[{k + 1}, size={min(card, n - card)}] \t {fnn.java_double_str(w[k])} \t {conf} \t  {members},"
    # everything else is the plain output
    stripped = [ln.replace("confidences=yes", "confidences=no") for ln in lines]
    for k in range(len(w)):
        head, wt, conf, rest = stripped[start + 1 + k].split(" \t ")
        stripped[start + 1 + k] = " \t ".join([head, wt, rest])
    assert "\n".join(stripped) == plain


def test_nexus_without_support_is_byte_identical(tmp_path):
    n = 12
    ordering = np.array([0] + list(range(n, 0, -1)), dtype=np.int32)
    si = np.array([0, 2, 4], dtype=np.int32)
    sj = np.array([3, 9, 11], dtype=np.int32)
    w = np.array([0.1, 0.2, 0.3])
    D = np.abs(np.subtract.outer(np.arange(n), np.arange(n))).astype(np.float64)
    ip = ctypes.POINTER(ctypes.c_int32)
    dp = ctypes.POINTER(ctypes.c_double)
    a, b = tmp_path / "a.nex", tmp_path / "b.nex"
    assert fnn.lib().fnn_write_nexus(str(a).encode(), n, None, 0, D.ctypes.data_as(dp), ordering.ctypes.data_as(ip),
                                     si.ctypes.data_as(ip), sj.ctypes.data_as(ip), w.ctypes.data_as(dp), 3, 1) == 0
    assert fnn.lib().fnn_write_nexus_support(str(b).encode(), n, None, 0, D.ctypes.data_as(dp), ordering.ctypes.data_as(ip),
                                             si.ctypes.data_as(ip), sj.ctypes.data_as(ip), w.ctypes.data_as(dp), None, 0, 3, 1) == 0
    assert a.read_bytes() == b.read_bytes()
    assert _nexus_text(tmp_path, "c.nex", ordering=ordering, split_i=si, split_j=sj, weight=w, D=D) == a.read_text()


def test_nexus_support_out_of_range_is_refused(tmp_path):
    ordering = np.arange(6, dtype=np.int32)
    with pytest.raises(fnn.FastNNError) as e:
        fnn.write_nexus(str(tmp_path / "x.nex"), ordering, [0], [2], [1.0], support=[4], replicates=3)
    assert e.value.code == -1 and "outside 0..3" in str(e.value)
    with pytest.raises(fnn.FastNNError):
        fnn.write_nexus(str(tmp_path / "x.nex"), ordering, [0], [2], [1.0], support=[0], replicates=0)


def test_cli_bootstrap_options():
    a = parse_args(["-seqFile", "x.fa", "-bootstrap", "20", "--bootstrap-seed", "7"])
    assert (a.bootstrap, a.bootstrap_seed) == (20, 7)
    assert parse_args(["-seqFile", "x.fa"]).bootstrap == 0
    for bad in (["-distFile", "x.phy", "-bootstrap", "5"], ["-seqFile", "x.fa", "-order", "-bootstrap", "5"],
                ["-seqFile", "x.fa", "-bootstrap", "-2"]):
        with pytest.raises(SystemExit):
            parse_args(bad)


def test_cli_bootstrap_error_messages(capsys):
    with pytest.raises(SystemExit):
        parse_args(["-distFile", "x.phy", "-bootstrap", "5"])
    assert "-bootstrap needs -seqFile" in capsys.readouterr().err
    with pytest.raises(SystemExit):
        parse_args(["-seqFile", "x.fa", "-order", "-bootstrap", "5"])
    assert "-order" in capsys.readouterr().err
