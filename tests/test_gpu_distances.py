"""GPU: alignment distances (fnn_distances, fnn_ctx_load_alignment) bit for bit against the CPU oracle (oracle/dist_oracle.cpp),
the context path into the ordering, and the -seqFile driver."""
import subprocess
import sys

import numpy as np
import pytest

import oracle
from oracle import dist as dist_oracle
from fastneighbornet_b200 import synth

pytestmark = pytest.mark.gpu

MODELS = ("p", "jc69", "k2p")


def _same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and (a.view(np.uint64) == b.view(np.uint64)).all()


def _random_codes(n, L, seed, missing=0.2):
    rng = np.random.default_rng(seed)
    c = rng.integers(0, 4, (n, L)).astype(np.uint8)
    c[rng.random((n, L)) < missing] = 4
    return c


def _check(fnn, codes, models=MODELS, undefined=None):
    for model in models:
        D = fnn.distances(codes, model=model, undefined=undefined)
        ref, first = dist_oracle.distances(codes, model, undefined=undefined)
        assert undefined is not None or first is None
        assert _same_bits(D, ref), (codes.shape, model)


@pytest.mark.parametrize("L", [1, 63, 64, 65, 1000, 4097])
@pytest.mark.parametrize("n", [1, 2, 4, 17, 127, 128, 129, 1000])
def test_sizes_random_and_simulated(fnn, n, L):
    # random codes saturate and have pairs without a comparable site: those entries get the substitute value
    _check(fnn, _random_codes(n, L, n * 10007 + L), undefined=3.5)
    _check(fnn, synth.simulate_alignment(n, L, n + L, rate=0.3, gap_frac=0.02), undefined=0.0)


def test_simulated_without_undefined_pairs(fnn):
    _check(fnn, synth.simulate_alignment(700, 2000, 7, rate=0.4, gap_frac=0.05))


def test_heavy_gaps_and_ambiguity(fnn):
    codes = synth.simulate_alignment(300, 1500, 8, gap_frac=0.85)
    _check(fnn, codes, undefined=1.25)
    _check(fnn, _random_codes(200, 700, 9, missing=0.95), undefined=0.0)


def test_identical_sequences(fnn):
    codes = np.tile(_random_codes(1, 777, 10), (150, 1))
    for model in MODELS:
        D = fnn.distances(codes, model=model)
        assert (D.view(np.uint64) == 0).all()   # +0.0 everywhere, no -0.0
        assert _same_bits(D, dist_oracle.distances(codes, model)[0])


def test_full_matrix_n3000_l5000(fnn):
    _check(fnn, synth.simulate_alignment(3000, 5000, 11, rate=0.4, gap_frac=0.05))


def test_n20000_l512_sampled_rows(fnn):
    n = 20000
    codes = synth.simulate_alignment(n, 512, 12, rate=0.3, gap_frac=0.05)
    rng = np.random.default_rng(13)
    tiles = rng.choice(np.arange(64, n, 64), 100, replace=False)   # both sides of 100 tile boundaries
    rows = np.unique(np.concatenate([[0, n - 1], tiles - 1, tiles, rng.choice(n, 298, replace=False)]))[:500]
    rows = np.unique(np.concatenate([rows[:498], [0, n - 1]]))
    for model in MODELS:
        D = fnn.distances(codes, model=model, undefined=2.0)
        ref, _ = dist_oracle.distances(codes, model, undefined=2.0, rows=rows)
        assert _same_bits(D[rows], ref), model
        assert _same_bits(D[:, rows].T, ref), model


def test_undefined_pairs(fnn):
    codes = _random_codes(300, 40, 14, missing=0.3)
    codes[5, :] = 4    # no comparable site with anyone
    for model in MODELS:
        _, first = dist_oracle.distances(codes, model)
        assert first is not None
        i, j, v, m, s = first
        with pytest.raises(fnn.FastNNError) as e:
            fnn.distances(codes, model=model)
        assert e.value.code == -1
        assert f"pair ({i}, {j})" in str(e.value) and f"v = {v} " in str(e.value) and f"m = {m} " in str(e.value) \
            and f"s = {s} " in str(e.value)
        with fnn.Context(300) as c:
            with pytest.raises(fnn.FastNNError) as e2:
                c.load_alignment(codes, model=model)
            assert str(e2.value) == str(e.value).replace("fnn_distances", "fnn_ctx_load_alignment")
            with pytest.raises(fnn.FastNNError) as e3:
                c.read_matrix()
            assert e3.value.code == -5   # left unloaded
        for sub in (0.0, 9.75):
            D = fnn.distances(codes, model=model, undefined=sub)
            assert _same_bits(D, dist_oracle.distances(codes, model, undefined=sub)[0])
            assert (D[5, np.arange(300) != 5] == sub).all()


def test_bad_codes_are_refused(fnn):
    codes = _random_codes(10, 100, 15)
    codes[3, 7] = 5
    with pytest.raises(fnn.FastNNError) as e:
        fnn.distances(codes, undefined=0.0)
    assert e.value.code == -1 and "outside 0..4" in str(e.value)


def test_context_path_and_ordering(fnn):
    n = 1000   # ld = 1008 > n
    codes = synth.simulate_alignment(n, 3000, 16, rate=0.3, gap_frac=0.05)
    for model in MODELS:
        D = fnn.distances(codes, model=model)
        with fnn.Context(n) as c:
            assert c.matrix_ptr()[1] > n
            c.load_alignment(codes, model=model)
            assert _same_bits(c.read_matrix(), D)
            st = c.stats()
            assert st["dist_pairs_ms"] > 0 and st["dist_pack_ms"] > 0 and st["h2d_ms"] > 0
        for mode in ("canonical", "relaxed"):
            with fnn.Context(n, mode=mode) as c:
                c.load_alignment(codes, model=model)
                o = c.order()
            assert (o == fnn.order(D, mode=mode)).all()
            o_ref, _, _ = oracle.order(D, mode=mode, want_trace=False)
            assert (o == o_ref).all(), (model, mode)


def test_driver_seqfile_equals_distfile(fnn, tmp_path):
    n = 60
    codes = synth.simulate_alignment(n, 900, 17, rate=0.3, gap_frac=0.05)
    names = [f"taxon{i}" for i in range(n)]
    fa = tmp_path / "aln.fa"
    synth.write_alignment(str(fa), codes, names)
    for model in ("p", "k2p"):
        phy = tmp_path / f"d_{model}.phy"
        synth.write_phylip(str(phy), fnn.distances(codes, model=model), names)
        for extra in ([], ["-order"]):
            r1 = subprocess.run([sys.executable, "-m", "fastneighbornet_b200", "-seqFile", str(fa), "--distance", model] + extra,
                                capture_output=True, text=True)
            r2 = subprocess.run([sys.executable, "-m", "fastneighbornet_b200", "-distFile", str(phy)] + extra,
                                capture_output=True, text=True)
            assert r1.returncode == 0 and r2.returncode == 0, r1.stderr + r2.stderr
            assert r1.stdout == r2.stdout and len(r1.stdout) > 0
