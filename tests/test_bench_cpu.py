"""CPU-only: the reference arm of bench.py (the CPU restatement of the reference, what the driver runs as `--impl reference`)
prints exactly one JSON line whose `config.n_taxa` is the size it really ran, with the 1-thread figure and the c*n^3 fit."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--ref-n", "300", "--fit-n", "300,450", "--fit-n1", "200,300"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GB/s" and d["higher_is_better"] is True and d["scaling"] == "strong"
    assert d["config"]["n_taxa"] == 300 and d["config"]["sample_of_n_taxa"] == 20000
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value_1thread"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    ex = d["extrapolated"]
    assert ex["extrapolated"] is True and ex["n_taxa"] == 20000
    assert ex["threads_all"]["fit_n"] == [300, 450] and ex["threads_all"]["seconds_at_workload_n"] > 0
    assert ex["threads_1"]["seconds_at_workload_n"] >= ex["threads_all"]["seconds_at_workload_n"] * 0.2


def test_reference_arm_dumps_last_step_ordering(tmp_path):
    """--dump-outputs writes what the last timed step computed: with --steps 2 that is the ordering of seed 2's matrix."""
    import numpy as np
    import oracle
    from fastneighbornet_b200 import synth
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0",
                        "--ref-n", "120", "--fit-n", "120", "--fit-n1", "100", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    got = np.load(tmp_path / "ordering.npy")
    assert got.dtype == np.float64
    o_ref, _, _ = oracle.order(synth.additive_noise_matrix(120, 2, 0.05), want_trace=False)
    assert (got == o_ref).all()


def test_zero_steps_is_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=60)
    assert r.returncode == 2 and "--steps" in r.stderr


def test_cubic_fit():
    sys.path.insert(0, ROOT)
    import bench
    c = bench.cubic_fit([1000, 2000, 4000], [2e-9 * n ** 3 for n in (1000, 2000, 4000)])
    assert abs(c - 2e-9) < 1e-15
