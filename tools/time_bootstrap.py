"""Time fnn_bootstrap on the GPU: where a replicate's time goes.

    python tools/time_bootstrap.py n L R [--model p|jc69|k2p] [--seed S]

Prints one JSON line: the CUDA-event ms per replicate of the four phases fnn_bootstrap measures (distances = packing + pair
kernels, ordering = fnn_ctx_order, split weights = triangle packing + solve + compaction, matching = support table +
k_support), the CG iterations per replicate, the host time of the whole call (original network included) per replicate,
and the card's name and power limit read in the same run.  The input is synth.simulate_alignment (seeded).
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fastneighbornet_b200 as fnn  # noqa: E402
from fastneighbornet_b200 import synth  # noqa: E402
from time_distances import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("n", type=int)
    ap.add_argument("L", type=int)
    ap.add_argument("R", type=int)
    ap.add_argument("--model", default="k2p", choices=list(fnn.MODELS))
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    if fnn.device_count() < 1:
        raise SystemExit("time_bootstrap: no CUDA device")
    codes = synth.simulate_alignment(a.n, a.L, a.seed, rate=0.3, gap_frac=0.02)
    fnn.bootstrap(codes[:, :64], 1, model=a.model, undefined=0.0)   # warm-up: module load, first launches
    t = time.perf_counter()
    b = fnn.bootstrap(codes, a.R, model=a.model, boot_seed=a.seed, undefined=0.0)
    wall = time.perf_counter() - t
    per = {k: round(v / a.R, 3) for k, v in b.times.items() if k.endswith("_ms")}
    out = {"n": a.n, "L": a.L, "R": a.R, "model": a.model, "card": card(), "per_replicate_ms": per,
           "cg_iters_per_replicate": b.times["cg_iters"] / a.R, "call_s_per_replicate": round(wall / a.R, 3),
           "call_s": round(wall, 2), "kept_splits": int(len(b.weight)),
           "mean_replicate_kept": float(b.replicate_kept.mean()), "mean_support": float(b.support.mean()) if len(b.support) else 0.0}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
