"""tools/time_order.py [--mode M] [--opt k=v ...] [--reps R] n [n ...] : wall time of one ordering per n (device-generated input)."""
import hashlib, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fastneighbornet_b200 as f
args = sys.argv[1:]
mode, opts, reps, eps = "canonical", {}, 1, 0.05
while args and args[0].startswith("--"):
    if args[0] == "--mode":
        mode = args[1]
    elif args[0] == "--opt":
        k, v = args[1].split("=")
        opts[k] = int(v)
    elif args[0] == "--reps":
        reps = int(args[1])
    elif args[0] == "--eps":
        eps = float(args[1])
    args = args[2:]
for n in [int(a) for a in args] or [5000, 20000]:
    with f.Context(n, mode=mode, **opts) as c:
        for r in range(reps):
            c.synth(1, eps)
            t = time.time(); o = c.order(); dt = time.time() - t
            s = c.stats()
            print(f"n={n} mode={mode} eps={eps} opts={opts} wall={dt:.3f}s dev={s['order_ms']/1e3:.3f}s iterations={s['iterations']} "
                  f"launches={s['kernel_launches']} alg={s['scan_alg_bytes']/dt/1e9:.0f} GB/s certified={s['picks_certified']} "
                  f"exact={s['picks_exact']} strat_units={s['strategy_units']} read={s['scan_read_bytes']/1e9:.1f} GB "
                  f"of alg={s['scan_alg_bytes']/1e9:.1f} GB skipped_units={s['scan_units_skipped']} "
                  f"sha={hashlib.sha256(o.tobytes()).hexdigest()[:16]}", flush=True)
