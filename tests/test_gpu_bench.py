"""GPU: bench.py --dump-outputs writes the ordering of the timed path's last step, and it is the oracle's ordering of the
seeded workload matrix."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from helpers import tree_matrix

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_is_the_timed_ordering(tmp_path):
    n = 1500
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--n", str(n), "--steps", "2", "--warmup", "1",
                        "--no-parity", "--no-e2e", "--no-configs", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout)
    assert line["steps"] == 2 and line["config"]["n_taxa"] == n
    got = np.load(tmp_path / "ordering.npy")
    assert got.dtype == np.float64 and got.shape == (n + 1,)
    o_ref, _, _ = oracle.order(tree_matrix(n, 1, 0.05), want_trace=False)   # bench.py's workload: seed 1, eps 0.05
    assert (got == o_ref).all()
