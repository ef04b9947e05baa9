"""CPU-only: the native alignment loader against a Python parser, its error cases, the shared logarithm fnn_log, the
distance oracle against an independent numpy count, and the alignment entry points failing loudly without a GPU."""
import subprocess
import sys
from decimal import Decimal, getcontext

import numpy as np
import pytest

import fastneighbornet_b200 as fnn
from oracle import dist as dist_oracle
from fastneighbornet_b200 import synth

CODE = {**{c: i for i, c in enumerate("ACGT")}, "U": 3, **{c: 4 for c in "RYSWKMBDHVNX-?"}}


def py_parse(path):
    """Independent reader of the two formats: (codes, names)."""
    text = open(path, "rb").read().decode("ascii")
    lines = text.replace("\r\n", "\n").split("\n")
    seqs, names = [], []
    if text.lstrip()[0] in ">;":
        for ln in lines:
            if ln.startswith(";"):
                continue
            if ln.startswith(">"):
                names.append(ln[1:].split()[0] if ln[1:].split() else "")
                seqs.append("")
            elif names:
                seqs[-1] += "".join(ln.split())
    else:
        body = [ln for ln in lines if ln.strip()]
        n, L = (int(t) for t in body[0].split())
        for ln in body[1:1 + n]:
            nm, *rest = ln.split()
            names.append(nm)
            seqs.append("".join(rest))
    codes = np.array([[CODE[ch.upper()] for ch in s] for s in seqs], dtype=np.uint8)
    return codes, names


def _write(tmp_path, name, text, mode="w"):
    p = tmp_path / name
    if mode == "wb":
        p.write_bytes(text)
    else:
        p.write_text(text)
    return str(p)


def _random_seqs(rng, n, L):
    alphabet = np.array(list("ACGTacgtUuRYSWKMBDHVNXrykmn-?"))
    return ["".join(rng.choice(alphabet, L)) for _ in range(n)]


@pytest.mark.parametrize("crlf", [False, True])
def test_fasta_matches_python_parser(tmp_path, crlf):
    rng = np.random.default_rng(3)
    seqs = _random_seqs(rng, 37, 211)
    out = ["; a comment line before the first record", ""]
    for i, s in enumerate(seqs):
        out.append(f">taxon_{i} some description {i}")
        k = 0
        while k < len(s):   # wrapped at varying widths, with blank and ';' lines and stray spaces inside
            w = int(rng.integers(1, 80))
            out.append(s[k:k + w] + (" " if rng.random() < 0.2 else ""))
            if rng.random() < 0.1:
                out.append("")
            if rng.random() < 0.05:
                out.append(";comment ACGT")
            k += w
    text = ("\r\n" if crlf else "\n").join(out) + "\n"
    p = _write(tmp_path, "a.fa", text)
    codes, names = fnn.read_alignment(p)
    ref, ref_names = py_parse(p)
    assert codes.dtype == np.uint8 and codes.shape == (37, 211)
    assert (codes == ref).all() and names == ref_names == [f"taxon_{i}" for i in range(37)]
    c1, n1 = fnn.read_alignment(p, threads=1)
    assert (c1 == codes).all() and n1 == names


@pytest.mark.parametrize("crlf", [False, True])
def test_phylip_matches_python_parser(tmp_path, crlf):
    rng = np.random.default_rng(4)
    seqs = _random_seqs(rng, 45, 97)
    out = ["45  97", ""]
    for i, s in enumerate(seqs):
        cut = int(rng.integers(0, len(s)))
        out.append(f"sp{i}\t{s[:cut]} {s[cut:]}")   # whitespace inside the sequence is skipped
        if rng.random() < 0.1:
            out.append("   ")
    text = ("\r\n" if crlf else "\n").join(out) + "\n"
    p = _write(tmp_path, "a.phy", text)
    codes, names = fnn.read_alignment(p)
    ref, ref_names = py_parse(p)
    assert codes.shape == (45, 97) and (codes == ref).all() and names == ref_names
    c1, n1 = fnn.read_alignment(p, threads=1)
    assert (c1 == codes).all() and n1 == names


def test_writers_round_trip_and_many_threads(tmp_path):
    codes = synth.simulate_alignment(300, 1000, 5, gap_frac=0.1)
    names = [f"n{i}" for i in range(300)]
    for fmt in ("fasta", "phylip"):
        p = str(tmp_path / f"x.{fmt}")
        synth.write_alignment(p, codes, names, fmt=fmt)
        for threads in (0, 1, 3):
            c, nm = fnn.read_alignment(p, threads=threads)
            assert (c == codes).all() and nm == names


def test_long_names_are_truncated(tmp_path):
    p = _write(tmp_path, "a.fa", ">" + "x" * 100 + "\nACGT\n>b\nAC-T\n")
    codes, names = fnn.read_alignment(p, name_len=16)
    assert names == ["x" * 15, "b"] and codes.tolist() == [[0, 1, 2, 3], [0, 1, 4, 3]]


ERRORS = [
    ("unequal.fa", ">a\nACGT\n>b\nACG\n", ["taxon 2 'b'", "line 3", "3 sites, expected 4"]),
    ("longer.fa", ">a\nACGT\n>b\nACGTA\n", ["taxon 2 'b'", "5 sites, expected 4"]),
    ("empty.fa", ">a\nACGT\n>b\n>c\nACGT\n", ["taxon 2 'b'", "empty sequence"]),
    ("empty_first.fa", ">a\n\n>b\nACGT\n", ["taxon 1 'a'", "empty sequence"]),
    ("none.fa", "; only a comment\n;\n", ["no sequences"]),
    ("blank.fa", "  \n\n", ["no sequences"]),
    ("dot.fa", ">a\nACGT\n>b\nAC.T\n", ["line 4, column 3", "'.'", "taxon 2 'b'"]),
    ("digit.fa", ">a\nAC\nG1\n", ["line 3, column 2", "'1'"]),
    ("protein.fa", ">a\nACGT\n>b\nACGT\n>c\nLEIF\n", ["line 6, column 1", "'L'", "taxon 3 'c'"]),
    ("unequal.phy", "2 4\na ACGT\nb ACG\n", ["taxon 2 'b'", "line 3", "3 sites, expected 4"]),
    ("empty.phy", "2 4\na ACGT\nb\n", ["taxon 2 'b'", "empty sequence"]),
    ("fewer.phy", "3 4\na ACGT\nb ACGT\n", ["header says 3 taxa", "2 sequence lines"]),
    ("more.phy", "1 4\na ACGT\nb ACGT\n", ["header says 1 taxa", "line 3"]),
    ("interleaved.phy", "2 8\na ACGT\nb ACGT\n\nACGT\nACGT\n", ["taxon 1 'a'", "4 sites, expected 8", "interleaved"]),
    ("none.phy", "0 4\n", ["no sequences"]),
    ("badheader.phy", "2 x\na AC\n", ["line 1", "PHYLIP header"]),
    ("protein.phy", "2 4\na ACGT\nb ACEF\n", ["line 3, column 5", "'E'"]),
    ("junk.txt", "hello\n", ["line 1", "'h'"]),
]


@pytest.mark.parametrize("name,text,parts", ERRORS, ids=[e[0] for e in ERRORS])
def test_error_cases(tmp_path, name, text, parts):
    p = _write(tmp_path, name, text)
    with pytest.raises(fnn.FastNNError) as e:
        fnn.read_alignment(p)
    assert e.value.code == -6, str(e.value)
    for part in parts:
        assert part in str(e.value), (part, str(e.value))


def test_error_names_the_first_bad_record_whatever_the_threads(tmp_path):
    seqs = ["ACGT" * 10] * 200
    seqs[150] = "ACGT" * 9 + "ACGE"
    seqs[170] = "ACG"
    p = _write(tmp_path, "x.fa", "".join(f">s{i}\n{s}\n" for i, s in enumerate(seqs)))
    for threads in (1, 0, 7):
        with pytest.raises(fnn.FastNNError) as e:
            fnn.read_alignment(p, threads=threads)
        assert "taxon 151 's150'" in str(e.value) and "'E'" in str(e.value)


def test_caller_size_mismatch_is_an_argument_error(tmp_path):
    import ctypes
    p = _write(tmp_path, "a.phy", "2 4\na ACGT\nb ACGT\n")
    buf = np.zeros(12, dtype=np.uint8)
    rc = fnn.lib().fnn_read_alignment(p.encode(), 3, 4, buf.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), None, 0, 0)
    assert rc == -1


# ---- fnn_log -----------------------------------------------------------------------------------------------------------

def _ulps(a, ref):
    return np.abs(a - ref) / np.spacing(np.abs(ref))


def _log_samples():
    rng = np.random.default_rng(11)
    x = np.concatenate([
        rng.random(500_000),
        np.exp(rng.uniform(-745.0, 0.0, 300_000)),
        rng.integers(1, 2 ** 52, 100_000).astype(np.float64) * 5e-324,    # subnormals
        np.ldexp(1.0, -np.arange(0, 1075)),                                  # powers of two down to 2^-1074
        1.0 - np.arange(1, 100_001) * 2.0 ** -53,                            # neighbours of 1
        np.nextafter(np.ldexp(1.0, -np.arange(1, 1022)), 0.0),
        np.nextafter(np.ldexp(1.0, -np.arange(1, 1022)), 1.0),
        np.ldexp(np.sqrt(0.5), -np.arange(0, 1000)),                        # the reduction boundary
    ])
    return x[(x > 0) & (x <= 1)]


def test_fnn_log_of_one_is_plus_zero():
    r = dist_oracle.fnn_log(np.array([1.0]))[0]
    assert r == 0.0 and not np.signbit(r)


def test_fnn_log_within_one_ulp_of_numpy_and_monotone():
    x = _log_samples()
    assert x.size >= 1_000_000
    y = dist_oracle.fnn_log(x)
    ref = np.log(x)
    assert np.isfinite(y).all()
    assert _ulps(y, ref).max() <= 1.0
    xs = np.sort(x)
    assert (np.diff(dist_oracle.fnn_log(xs)) >= 0).all()
    special = dist_oracle.fnn_log(np.array([0.0, -1.0, np.inf, np.nan, 2.0, 1e300]))
    assert special[0] == -np.inf and np.isnan(special[1]) and special[2] == np.inf and np.isnan(special[3])
    assert _ulps(special[4:], np.log([2.0, 1e300])).max() <= 1.0


def test_fnn_log_within_one_ulp_of_a_decimal_log():
    getcontext().prec = 40
    x = _log_samples()
    x = x[np.random.default_rng(2).choice(x.size, 3000, replace=False)]
    y = dist_oracle.fnn_log(x)
    for xi, yi in zip(x, y):
        exact = Decimal(float(xi)).ln()
        err = abs(Decimal(float(yi)) - exact) / Decimal(float(np.spacing(abs(float(exact)))))
        assert err <= 1, (xi, yi, exact)


# ---- the distance oracle against an independent numpy count -------------------------------------------------------------

def numpy_counts(codes):
    c = codes.astype(np.int64)
    oh = [(c == k).astype(np.int64) for k in range(4)]
    ok = sum(oh)
    v = ok @ ok.T
    same = sum(o @ o.T for o in oh)
    s = oh[0] @ oh[2].T + oh[2] @ oh[0].T + oh[1] @ oh[3].T + oh[3] @ oh[1].T
    return v, v - same, s


def numpy_distances(codes, model, undefined=None):
    """The formulas of include/fastnn.h in numpy, over the numpy counts; logs through the shared fnn_log."""
    v, m, s = numpy_counts(codes)
    n = codes.shape[0]
    with np.errstate(divide="ignore", invalid="ignore"):
        dv = v.astype(np.float64)
        if model == "p":
            D = m / dv
            undef = v == 0
        elif model == "jc69":
            arg = 1.0 - (m / dv) / 0.75
            undef = (v == 0) | ~(arg > 0)
            D = -0.75 * dist_oracle.fnn_log(np.where(undef, 1.0, arg))
        else:
            P, Q = s / dv, (m - s) / dv
            a1, a2 = (1.0 - 2.0 * P) - Q, 1.0 - 2.0 * Q
            undef = (v == 0) | ~(a1 > 0) | ~(a2 > 0)
            D = (-0.5 * dist_oracle.fnn_log(np.where(undef, 1.0, a1))) - (0.25 * dist_oracle.fnn_log(np.where(undef, 1.0, a2)))
    D = np.where(D == 0.0, 0.0, D)
    np.fill_diagonal(undef, False)
    D[undef] = np.nan if undefined is None else undefined
    np.fill_diagonal(D, 0.0)
    iu = np.argwhere(np.triu(undef, 1))
    first = None
    if len(iu):
        i, j = (int(t) for t in iu[0])
        first = (i, j, int(v[i, j]), int(m[i, j]), int(s[i, j]))
    return D, first


def _same_bits(a, b):
    return a.shape == b.shape and (a.view(np.uint64) == b.view(np.uint64)).all()


CASES = {
    "random": lambda: np.random.default_rng(1).integers(0, 5, (23, 300)).astype(np.uint8),
    "simulated": lambda: synth.simulate_alignment(40, 700, 2, rate=0.4, gap_frac=0.05),
    "heavy_gaps": lambda: synth.simulate_alignment(30, 200, 3, gap_frac=0.7),
    "identical": lambda: np.tile(np.random.default_rng(4).integers(0, 5, 129).astype(np.uint8), (9, 1)),
    "short": lambda: np.random.default_rng(5).integers(0, 5, (17, 3)).astype(np.uint8),
}


@pytest.mark.parametrize("model", list(fnn.MODELS))
@pytest.mark.parametrize("case", list(CASES))
def test_oracle_matches_numpy(case, model):
    codes = CASES[case]()
    for undefined in (None, 0.5, 0.0):
        D, first = dist_oracle.distances(codes, model, undefined=undefined)
        ref, ref_first = numpy_distances(codes, model, undefined)
        assert _same_bits(D, ref), (case, model, undefined)
        assert first == ref_first
        assert not np.signbit(D[~np.isnan(D)]).any()
        assert _same_bits(D, np.ascontiguousarray(D.T))
    rows = np.array([codes.shape[0] - 1, 0, 2 % codes.shape[0]])
    Dr, _ = dist_oracle.distances(codes, model, undefined=0.25, rows=rows)
    full, _ = dist_oracle.distances(codes, model, undefined=0.25)
    assert _same_bits(Dr, full[rows])


def test_oracle_minus_zero_saturation_and_first_undefined():
    # taxa 0 and 1 identical (m = 0: JC69 and K2P give -0.75*log(1) = -0.0, stored +0.0); taxa 0 and 2 differ at every site
    # (saturated under JC69 and K2P), taxon 3 has no state at all (v = 0 with everyone)
    codes = np.array([[0, 1, 2, 3] * 4, [0, 1, 2, 3] * 4, [1, 0, 3, 2] * 4, [4] * 16], dtype=np.uint8)
    for model in ("jc69", "k2p"):
        D, first = dist_oracle.distances(codes, model)
        assert D[0, 1] == 0.0 and not np.signbit(D[0, 1])
        assert np.isnan(D[0, 2]) and first == (0, 2, 16, 16, 0)
        D5, _ = dist_oracle.distances(codes, model, undefined=5.0)
        assert D5[0, 2] == 5.0 and D5[2, 0] == 5.0 and (D5[3, :3] == 5.0).all() and D5[3, 3] == 0.0
    D, first = dist_oracle.distances(codes, "p")
    assert D[0, 2] == 1.0 and first == (0, 3, 0, 0, 0)


# ---- no GPU ------------------------------------------------------------------------------------------------------------

@pytest.mark.skipif(fnn.device_count() > 0, reason="GPU present")
def test_alignment_entry_points_fail_loudly_without_gpu(tmp_path):
    codes = synth.simulate_alignment(6, 50, 1)
    with pytest.raises(fnn.FastNNError) as e:
        fnn.distances(codes, model="k2p")
    assert e.value.code == -2 and "no CPU fallback" in str(e.value)
    with pytest.raises(fnn.FastNNError) as e:
        with fnn.Context(6) as c:
            c.load_alignment(codes)
    assert e.value.code == -2
    p = tmp_path / "a.fa"
    synth.write_alignment(str(p), codes)
    r = subprocess.run([sys.executable, "-m", "fastneighbornet_b200", "-seqFile", str(p), "-order"], capture_output=True, text=True)
    assert r.returncode == 2 and "no CUDA device" in r.stderr and r.stdout == ""


def test_distance_arguments_are_checked_before_the_device():
    codes = synth.simulate_alignment(4, 10, 1)
    for bad in (-1.0, float("inf"), -float("inf")):
        with pytest.raises(fnn.FastNNError) as e:
            fnn.distances(codes, undefined=bad)
        assert e.value.code == -1
    with pytest.raises(ValueError):
        fnn.distances(codes, model="f81")
    with pytest.raises(fnn.FastNNError) as e:
        fnn.distances(np.zeros((3, 0), dtype=np.uint8))
    assert e.value.code == -1


def test_cli_options():
    from fastneighbornet_b200.__main__ import parse_args
    a = parse_args(["-seqFile", "x.fa", "--distance", "k2p", "--undefined", "2.5"])
    assert (a.seqFile, a.distFile, a.distance, a.undefined) == ("x.fa", None, "k2p", 2.5)
    assert parse_args(["-seqFile", "x.fa"]).distance == "p" and parse_args(["-seqFile", "x.fa"]).undefined is None
    with pytest.raises(SystemExit):
        parse_args(["-seqFile", "x.fa", "-distFile", "x.phy"])
    with pytest.raises(SystemExit):
        parse_args(["-seqFile", "x.fa", "--distance", "f81"])
