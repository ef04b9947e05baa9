"""`python -m fastneighbornet_b200 -distFile in.phy | -seqFile aln.fa [...]` — the run of FastNN.main (FastNN.java:113-480) over libfastnn.so.

A thin driver, kept only so that the three native stages can be exercised the way the reference is invoked:
fnn_read_phylip -> fnn_network (ordering, split weights, kept splits; distances stay on the device) -> fnn_write_nexus.
-seqFile replaces the first stage with fnn_read_alignment -> fnn_distances (--distance p|jc69|k2p, --undefined VALUE).
Options carry the reference's names (FastNN.java:130-172); -threads is accepted and only sizes the host-side loader and
writer pools.  --seed is new: the reference draws from an unseedable ThreadLocalRandom in the Relaxed/Random modes.
"""
import argparse
import sys
import time

import numpy as np

from . import api

MODES = {"CANONICAL": "canonical", "RELAXED": "relaxed", "RANDOM_N": "random_n", "RANDOM_NLOGN": "random_nlogn", "RANDOM_LOGN": "random_logn"}


def parse_args(argv):
    ap = argparse.ArgumentParser(prog="python -m fastneighbornet_b200", prefix_chars="-", allow_abbrev=False,
                                 description="Neighbor-Net on a B200: circular ordering and weighted splits as Nexus on stdout.")
    src = ap.add_mutually_exclusive_group(required=True)
    src.add_argument("-distFile", metavar="file_location", help="Phylip distance matrix (lower-triangular or square)")
    src.add_argument("-seqFile", metavar="file_location",
                     help="nucleotide alignment (FASTA or sequential PHYLIP); distances are computed on the GPU")
    ap.add_argument("-threads", type=int, default=0, metavar="integer", help="host threads for the loader/writer (0 = all)")
    ap.add_argument("-mode", default="CANONICAL", metavar="string", help="|".join(MODES))
    ap.add_argument("-mult", type=int, default=5, metavar="integer", help="multiplier of the Random_* sample sizes")
    ap.add_argument("-order", action="store_true", help="Outputs the circular order only.")
    ap.add_argument("-additive", action="store_true", help="Performs an additivity check for the relaxed search strategy.")
    ap.add_argument("-time", action="store_true", help="Show timing results.")
    ap.add_argument("--seed", type=int, default=12345)
    ap.add_argument("--no-distances", action="store_true", help="leave the n x n Distances block out of the Nexus output")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--distance", default="p", choices=list(api.MODELS), help="distance model of -seqFile (default p)")
    ap.add_argument("--undefined", type=float, default=None, metavar="VALUE",
                    help="-seqFile: distance of a pair with no comparable site or a saturated one (default: such a pair is an error)")
    a = ap.parse_args(argv)
    if a.mode.upper() not in MODES:
        ap.error(f"-mode must be one of {', '.join(MODES)}")
    a.mode = MODES[a.mode.upper()]
    return a


def main(argv=None):
    a = parse_args(sys.argv[1:] if argv is None else argv)
    t0 = time.perf_counter()
    if a.seqFile:
        codes, names = api.read_alignment(a.seqFile, threads=a.threads)
        D = api.distances(codes, model=a.distance, undefined=a.undefined, device=a.device)
    else:
        D, names = api.read_phylip(a.distFile, threads=a.threads)
    n = D.shape[0]
    t1 = time.perf_counter()
    print(f"Calculating a network for {n} taxa on CUDA device {a.device}.", file=sys.stderr)
    opts = dict(mode=a.mode, mult=a.mult, additive=a.additive, seed=a.seed, device=a.device)
    if a.order or n < 4:
        ordering = api.order(D, **opts)
        t2 = time.perf_counter()
        if a.order:
            print("[" + ", ".join(str(int(v)) for v in ordering) + "]")     # Arrays.toString(ordering), FastNN.java:395
        else:
            api.write_nexus(None, ordering, [], [], [], D=None if a.no_distances else D, names=names, threads=a.threads)
        sys.stdout.flush()
        if a.time:
            print(f"load {t1 - t0:.3f} s, ordering {t2 - t1:.3f} s", file=sys.stderr)
        return 0
    ordering, si, sj, w = api.network(D, **opts)
    t2 = time.perf_counter()
    sys.stdout.flush()
    api.write_nexus(None, ordering, si, sj, w, D=None if a.no_distances else D, names=names, threads=a.threads)
    t3 = time.perf_counter()
    if a.time:
        print(f"load {t1 - t0:.3f} s, ordering + split weights {t2 - t1:.3f} s, output {t3 - t2:.3f} s; {len(w)} splits kept", file=sys.stderr)
    return 0


if __name__ == "__main__":
    try:
        sys.exit(main())
    except api.FastNNError as e:
        print(f"fastneighbornet_b200: {e}", file=sys.stderr)
        sys.exit(2)
