"""GPU: fnn_bootstrap held exactly to the CPU composition of the oracles (tests/boot_oracle.py): the original network, every
replicate's ordering and kept-split count, and the support counts; the original network against fnn_network(fnn_distances);
undefined pairs in a replicate; seeds; and the -bootstrap driver."""
import subprocess
import sys

import numpy as np
import pytest

import boot_oracle
import oracle
from fastneighbornet_b200 import synth

pytestmark = pytest.mark.gpu

MODELS = ("p", "jc69", "k2p")


def _undefined_at(ref):
    """(replicate index or None for the original, (i, j, v, m, s)) of the first undefined pair of the oracle run, or None."""
    if "undefined" in ref["original"]:
        return None, ref["original"]["undefined"]
    for r, rep in enumerate(ref["replicates"]):
        if "undefined" in rep:
            return r, rep["undefined"]
    return None


def _compare(fnn, codes, R, boot_seed, model, undefined=None, mode="canonical", seed=12345, fallback=1024):
    ref = boot_oracle.bootstrap(codes, R, boot_seed, model=model, undefined=undefined, mode=mode, seed=seed, fallback=fallback)
    kw = dict(model=model, boot_seed=boot_seed, undefined=undefined, replicate_orderings=True, mode=mode, seed=seed,
              canonical_fallback=fallback)
    bad = _undefined_at(ref) if undefined is None else None
    if bad is not None:
        with pytest.raises(fnn.FastNNError) as e:
            fnn.bootstrap(codes, R, **kw)
        r, (i, j, v, m, s) = bad
        where = "" if r is None else f"replicate {r}: "
        assert e.value.code == -1
        assert f"fnn_bootstrap: {where}the {model} distance of pair ({i}, {j}) is undefined: v = {v} comparable sites, m = {m} " \
               f"differences, s = {s} transitions" in str(e.value)
        return None, ref
    b = fnn.bootstrap(codes, R, **kw)
    o = ref["original"]
    assert (b.ordering == o["ordering"]).all()
    assert (b.split_i == o["split_i"]).all() and (b.split_j == o["split_j"]).all()
    assert (b.weight.view(np.uint64) == o["weight"].view(np.uint64)).all()
    assert len(ref["replicates"]) == R
    for r, rep in enumerate(ref["replicates"]):
        assert (b.replicate_orderings[r] == rep["ordering"]).all(), r
        assert b.replicate_kept[r] == len(rep["weight"]), r
    assert b.support.dtype == np.int32 and (b.support == ref["support"]).all()
    assert ((b.support >= 0) & (b.support <= R)).all()
    assert b.times["cg_iters"] == sum(rep["cg_iters"] for rep in ref["replicates"])
    return b, ref


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("L", [64, 1000, 2001])
@pytest.mark.parametrize("n", [4, 5, 33, 64, 65, 130])
def test_against_oracle(fnn, n, L, model):
    R = 8 if n >= 100 else (12 if n >= 60 else 20)
    codes = synth.simulate_alignment(n, L, n * 1009 + L, rate=0.3, gap_frac=0.05)
    # L = 64 resamples can leave a pair without a comparable site or saturated: there the substitute is used
    b, ref = _compare(fnn, codes, R, n + L, model, undefined=2.0 if L == 64 else None)
    if b is not None:
        assert len(b.weight) > 0


@pytest.mark.parametrize("mode", ["relaxed", "random_nlogn"])
def test_other_orderings_against_oracle(fnn, mode):
    codes = synth.simulate_alignment(130, 1000, 21, rate=0.3, gap_frac=0.05)
    b, _ = _compare(fnn, codes, 6, 22, "k2p", mode=mode, seed=99, fallback=16)
    assert b is not None


def test_original_is_the_network_of_the_distances(fnn):
    codes = synth.simulate_alignment(90, 1500, 23, rate=0.3, gap_frac=0.05)
    for model in MODELS:
        b = fnn.bootstrap(codes, 3, model=model, boot_seed=5)
        o, si, sj, w = fnn.network(fnn.distances(codes, model=model))
        assert (b.ordering == o).all() and (b.split_i == si).all() and (b.split_j == sj).all()
        assert (b.weight.view(np.uint64) == w.view(np.uint64)).all()


def test_several_support_blocks_n300(fnn):
    """n = 300: about 700 kept splits per replicate, so k_support runs several blocks.  Every replicate is recomputed
    through fnn_network(fnn_distances(resampled columns)), and the support is counted by brute force on taxon sets."""
    n, L, R, seed = 300, 1000, 3, 24
    codes = synth.simulate_alignment(n, L, 25, rate=0.3, gap_frac=0.05)
    b = fnn.bootstrap(codes, R, model="k2p", boot_seed=seed, replicate_orderings=True)
    assert len(b.weight) > 256
    draws = oracle.java_random(seed, L, R * L).reshape(R, L)
    index = {boot_oracle.split_key(n, b.ordering[i + 1: j + 1]): k for k, (i, j) in enumerate(zip(b.split_i, b.split_j))}
    support = np.zeros(len(index), dtype=np.int32)
    for r in range(R):
        o, si, sj, _ = fnn.network(fnn.distances(codes[:, np.sort(draws[r])], model="k2p"))
        assert (b.replicate_orderings[r] == o).all() and b.replicate_kept[r] == len(si)
        assert len(si) > 256
        for i, j in zip(si, sj):
            k = index.get(boot_oracle.split_key(n, o[i + 1: j + 1]))
            if k is not None:
                support[k] += 1
    assert (b.support == support).all()


def test_constant_columns_give_full_support(fnn):
    rng = np.random.default_rng(26)
    col = rng.integers(0, 4, 40).astype(np.uint8)
    codes = np.repeat(col[:, None], 500, axis=1)   # every resample is the same alignment
    R = 9
    b = fnn.bootstrap(codes, R, model="p", boot_seed=27, replicate_orderings=True)
    assert (b.support == R).all()
    assert (b.replicate_orderings == b.ordering).all() and (b.replicate_kept == len(b.weight)).all()
    _compare(fnn, codes, R, 27, "p")


def _gappy(n, L, seed):
    codes = synth.simulate_alignment(n, L, seed, rate=0.2, gap_frac=0.05)
    codes[:, 0] = 2    # one column without a gap or a difference
    codes[:2, 1:] = 4  # taxa 0 and 1 have nothing else: a replicate without column 0 leaves them no comparable site
    return codes


@pytest.mark.parametrize("model", ["p", "k2p"])
def test_gap_heavy_undefined_pairs(fnn, model):
    codes = _gappy(33, 64, 28)
    R = 20
    _, ref = _compare(fnn, codes, R, 29, model)
    r, first = _undefined_at(ref)
    assert r is not None, "the oracle found no replicate with an undefined pair"
    if (ref["draws"][r] != 0).all():
        assert first[:2] == (0, 1) and first[2] == 0
    for sub in (0.0, 1.5):
        _compare(fnn, codes, R, 29, model, undefined=sub)


def test_seeds(fnn):
    codes = synth.simulate_alignment(33, 1000, 30, rate=0.3, gap_frac=0.05)
    a = fnn.bootstrap(codes, 10, boot_seed=31, replicate_orderings=True)
    b = fnn.bootstrap(codes, 10, boot_seed=31, replicate_orderings=True)
    c = fnn.bootstrap(codes, 10, boot_seed=32, replicate_orderings=True)
    for f in ("ordering", "split_i", "split_j", "support", "replicate_kept", "replicate_orderings"):
        assert (getattr(a, f) == getattr(b, f)).all(), f
    assert (a.weight.view(np.uint64) == b.weight.view(np.uint64)).all()
    assert (a.ordering == c.ordering).all() and (a.weight == c.weight).all()   # the original does not depend on the seed
    assert not (oracle.java_random(31, 1000, 10000) == oracle.java_random(32, 1000, 10000)).all()
    assert not ((a.support == c.support).all() and (a.replicate_kept == c.replicate_kept).all()
                and (a.replicate_orderings == c.replicate_orderings).all())


def test_driver_writes_confidences(fnn, tmp_path):
    n, R = 40, 20
    codes = synth.simulate_alignment(n, 800, 33, rate=0.3, gap_frac=0.05)
    fa = tmp_path / "aln.fa"
    synth.write_alignment(str(fa), codes, [f"taxon{i}" for i in range(n)])
    r = subprocess.run([sys.executable, "-m", "fastneighbornet_b200", "-seqFile", str(fa), "-bootstrap", str(R), "--bootstrap-seed", "34",
                        "-time"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "bootstrap, 20 replicates" in r.stderr
    b = fnn.bootstrap(codes, R, boot_seed=34)
    lines = r.stdout.split("\n")
    assert "FORMAT labels=no weights=yes confidences=yes intervals=no;" in lines
    start = lines.index("MATRIX", lines.index("BEGIN Splits;"))
    conf = [float(lines[start + 1 + k].split(" \t ")[2]) for k in range(len(b.weight))]
    assert conf == [100.0 * s / R for s in b.support]
    assert lines[start + 1 + len(b.weight)] == ";"
