"""Time Context.load_alignment (distances of an n x L alignment into the context's matrix) on the GPU.

    python tools/time_distances.py n L [--model p|jc69|k2p] [--reps R]

Reports the CUDA-event times the library records for the upload of the codes, the packing kernel and the pair kernel
(fnn_ctx_stats after fnn_ctx_load_alignment), the host time of the whole call, the word rate n(n-1)/2 * ceil(L/64) per second
and the 64-bit popcount rate of the pair kernel (2 per pair and word for p / jc69, 3 for k2p), with the card's name and
power limit read in the same run.  One warm-up call, then R timed calls.  The input is synth.simulate_alignment (seeded).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fastneighbornet_b200 as fnn  # noqa: E402
from fastneighbornet_b200 import synth  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = "unknown"
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("n", type=int)
    ap.add_argument("L", type=int)
    ap.add_argument("--model", default="p", choices=list(fnn.MODELS))
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    if fnn.device_count() < 1:
        raise SystemExit("time_distances: no CUDA device")
    t0 = time.perf_counter()
    codes = synth.simulate_alignment(a.n, a.L, 1, rate=0.3, gap_frac=0.02)
    gen_s = time.perf_counter() - t0
    words = (a.L + 63) // 64
    pair_words = a.n * (a.n - 1) / 2 * words
    popc = pair_words * (3 if a.model == "k2p" else 2)
    rows = []
    with fnn.Context(a.n) as c:
        for rep in range(a.reps + 1):
            t = time.perf_counter()
            c.load_alignment(codes, model=a.model, undefined=0.0)
            wall = (time.perf_counter() - t) * 1e3
            st = c.stats()
            if rep:
                rows.append((st["h2d_ms"], st["dist_pack_ms"], st["dist_pairs_ms"], wall))
    r = np.array(rows)
    med = np.median(r, axis=0)
    out = {
        "n": a.n, "L": a.L, "model": a.model, "reps": a.reps, "card": card(),
        "upload_ms": round(float(med[0]), 3), "pack_ms": round(float(med[1]), 3), "pairs_ms": round(float(med[2]), 3),
        "call_ms": round(float(med[3]), 3), "pairs_ms_min_max": [round(float(r[:, 2].min()), 3), round(float(r[:, 2].max()), 3)],
        "pair_words_per_s": pair_words / (med[2] * 1e-3), "popc64_per_s": popc / (med[2] * 1e-3),
        "simulate_alignment_s": round(gen_s, 1),
    }
    print(json.dumps(out))


if __name__ == "__main__":
    main()
