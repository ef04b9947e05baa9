"""Synthetic Phylip inputs: random additive tree metrics plus symmetric multiplicative noise.

Counter-based so the device generator (csrc/synth.cu, `fnn_synth_device`) produces the
same bits: every random number is splitmix64 of an integer key.

    h_k  = u01(S1 + k)            k < n-1   separator heights between DFS slots k, k+1
    a_i  = 0.5 * u01(S2 + i)      i < n     pendant lengths per DFS slot
    pi   = Fisher-Yates on hashes S4 + k    DFS slot -> taxon (0-based)
    d(pi(i), pi(j)) = ((2*max(h_i..h_{j-1}) + a_i) + a_j) * (1 + eps*(2*u01(S3 + lo*n + hi) - 1)),  i<j
      with lo<hi the two taxon indices.  eps = 0 gives an exact additive tree metric.

SURVEY.md §8(d) "Synthetic inputs".
"""
import numpy as np

_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def splitmix64(x):
    """Vectorised splitmix64 finaliser on uint64 arrays (wraps mod 2^64)."""
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = x + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def u01(keys):
    return (splitmix64(keys) >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def stream_base(seed, stream):
    return int(splitmix64(np.uint64((int(seed) * 8 + stream) & 0xFFFFFFFFFFFFFFFF)))


def tree_params(n, seed):
    """O(n) host-side parameters shared by the numpy and the device generator."""
    s1, s2, s4 = stream_base(seed, 1), stream_base(seed, 2), stream_base(seed, 4)
    with np.errstate(over="ignore"):
        k = np.arange(n, dtype=np.uint64)
        h = u01(np.uint64(s1) + k[: max(n - 1, 0)])
        a = 0.5 * u01(np.uint64(s2) + k)
        r = splitmix64(np.uint64(s4) + k)
    pi = np.arange(n, dtype=np.int64)
    for i in range(n - 1, 0, -1):  # Fisher-Yates
        j = int(r[i] % np.uint64(i + 1))
        pi[i], pi[j] = pi[j], pi[i]
    inv = np.empty(n, dtype=np.int64)
    inv[pi] = np.arange(n, dtype=np.int64)
    return h, a, pi, inv


def additive_noise_matrix(n, seed, eps=0.05):
    """n x n float64 symmetric distance matrix, zero diagonal (host, numpy)."""
    h, a, pi, inv = tree_params(n, seed)
    s3 = np.uint64(stream_base(seed, 3))
    M = np.zeros((n, n), dtype=np.float64)  # DFS-slot space
    for i in range(n - 1):
        mx = np.maximum.accumulate(h[i:])  # mx[t] = max(h_i..h_{i+t}) -> pair (i, i+t+1)
        row = (2.0 * mx + a[i]) + a[i + 1:]
        M[i, i + 1:] = row
        M[i + 1:, i] = row
    D = M[np.ix_(inv, inv)]  # D[t1][t2] = M[slot(t1)][slot(t2)]
    if eps != 0.0:
        with np.errstate(over="ignore"):
            for t in range(n):
                hi = np.arange(t + 1, n, dtype=np.uint64)
                keys = s3 + np.uint64(t) * np.uint64(n) + hi
                f = 1.0 + eps * (2.0 * u01(keys) - 1.0)
                v = D[t, t + 1:] * f
                D[t, t + 1:] = v
                D[t + 1:, t] = v
    return np.ascontiguousarray(D)


def upper_triangle(D):
    """Packed upper triangle in DistancesAndNames order (DistancesAndNames.java:24-38)."""
    n = D.shape[0]
    iu = np.triu_indices(n, 1)
    return np.ascontiguousarray(D[iu])


def write_phylip(path, D, names=None):
    """Lower-triangular Phylip as consumed by DistancesAndNames.java:43-132 (17 significant digits)."""
    n = D.shape[0]
    with open(path, "w") as f:
        f.write(f"{n}\n")
        for i in range(n):
            nm = names[i] if names is not None else f"t{i + 1}"
            f.write(nm)
            for j in range(i):
                f.write(" " + repr(float(D[i, j])))
            f.write("\n")


def read_phylip(path):
    """Reader with the reference's conventions: first line n; `name v v v ...`; only columns < row
    are consumed, so square and lower-triangular files both work (DistancesAndNames.java:63-107)."""
    with open(path) as f:
        n = int("".join(f.readline().split()))
        D = np.zeros((n, n), dtype=np.float64)
        names = []
        row = 0
        for line in f:
            ss = line.rstrip("\n").split(" ")
            if not ss or ss[0] == "" and len(ss) == 1:
                break
            names.append(ss[0])
            vals = []
            for tok in ss[1:]:
                if tok.strip():
                    vals.extend(tok.split("\t"))
            for col in range(row):
                D[row, col] = D[col, row] = float(vals[col])
            row += 1
            if row == n:
                break
    return D, names


# ---- nucleotide alignments (A=0 C=1 G=2 T=3, 4 = missing; the codes of api.read_alignment) ----------------------------

def simulate_alignment(n, L, seed, rate=0.3, gap_frac=0.0, kappa=2.0):
    """n x L uint8 alignment evolved under K2P along a random tree (seeded numpy).

    The tree is a random recursive tree: taxon k > 0 descends from a uniformly drawn earlier taxon over a branch of length
    Exp(1) * rate / max(1, ln n) substitutions per site, so a tip lies about `rate` substitutions from taxon 0 whatever n is
    and pairs stay far from saturation for rate <= 0.5.  Along a branch of length t each site takes a transition with
    probability 1/4 + e^(-4 b t)/4 - e^(-2 (a + b) t)/2 and one of the two transversions with probability 1/2 - e^(-4 b t)/2,
    with a = kappa / (kappa + 2), b = 1 / (kappa + 2).  A fraction gap_frac of the entries, drawn uniformly, is then set
    missing."""
    rng = np.random.default_rng(seed)
    codes = np.empty((n, L), dtype=np.uint8)
    codes[0] = rng.integers(0, 4, L, dtype=np.uint8)
    a, b = kappa / (kappa + 2.0), 1.0 / (kappa + 2.0)
    scale = rate / max(1.0, float(np.log(n)))
    parents = np.concatenate([[0], [int(rng.integers(0, k)) for k in range(1, n)]]) if n > 1 else np.zeros(1, dtype=np.int64)
    lengths = rng.exponential(scale, n)
    flip = np.array([1, 3], dtype=np.uint8)
    for k in range(1, n):
        t = lengths[k]
        p_ts = 0.25 + 0.25 * np.exp(-4 * b * t) - 0.5 * np.exp(-2 * (a + b) * t)
        p_tv = 0.5 - 0.5 * np.exp(-4 * b * t)
        u = rng.random(L)
        x = codes[parents[k]].copy()
        ts = u < p_ts
        tv = (u >= p_ts) & (u < p_ts + p_tv)
        x[ts] ^= 2
        x[tv] ^= flip[rng.integers(0, 2, int(tv.sum()))]
        codes[k] = x
    if gap_frac > 0:
        codes[rng.random((n, L)) < gap_frac] = 4
    return codes


def write_alignment(path, codes, names=None, fmt="fasta", width=60):
    """FASTA (sequences wrapped at `width`) or sequential relaxed PHYLIP (`n L`, then `name sequence` lines) of a code array;
    missing data is written as '-'."""
    n, L = codes.shape
    letters = np.frombuffer(b"ACGT-", dtype=np.uint8)
    with open(path, "w") as f:
        if fmt == "phylip":
            f.write(f"{n} {L}\n")
        for i in range(n):
            nm = names[i] if names is not None else f"t{i + 1}"
            seq = letters[codes[i]].tobytes().decode()
            if fmt == "phylip":
                f.write(f"{nm} {seq}\n")
            else:
                f.write(f">{nm}\n")
                for s in range(0, L, width):
                    f.write(seq[s:s + width] + "\n")
