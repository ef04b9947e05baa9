#!/usr/bin/env python
"""bench.py — the driver's measurement contract for the Neighbor-Net hot path.

A "step" is one full canonical Neighbor-Net ordering (NetMakerOriginal.runNeighborNet,
/root/reference NetMakerOriginal.java:129) of a synthetic n-taxon matrix (additive tree + 5 %
noise, SURVEY §8d).  metric/unit: algorithmic HBM GB/s of the job = the selection scan's
algorithmic bytes (8 B per cross-cluster matrix entry per iteration, SURVEY §8d; summed exactly
on the device) divided by the wall time of the whole ordering, so it is comparable across n and
between the GPU and the CPU arms; `ms_per_step` is the ordering's wall time.

  value     inputs resident in HBM (device matrix restored from a pristine device copy each step)
  e2e       the same through the reference-facing one-shot C-ABI call fnn_order() with a pinned
            HOST matrix: H2D of n*n*8 bytes + ordering + D2H of the ordering, all timed
  roofline  the selection kernel k_scan_tma: algorithmic bytes per launch / CUDA-event launch time,
            sampled every 16th iteration inside a dedicated profiled run of the same workload
  parity    BEFORE the timed region, at the SAME world size: orderings (and per-iteration traces) of
            n=1500 and n=5000 (> the 4096-node sharding threshold) against the CPU oracle, plus the
            sha256 of the n=20000 ordering (N>1 lines also carry the hash of an un-wired 1-GPU run)
  configs   one timed run each of the other BASELINE configs that fit the step budget (N=1 only)
  cpu_baseline / --impl reference: the CPU restatement of the reference (oracle/, "port": the JAR
            cannot run here - no JVM) on bounded samples, all host threads and 1 thread, with the
            c*n^3 fit that extrapolates the CPU wall time to the workload's n.
  --dump-outputs DIR  the ordering the timed path returned in its last step, as DIR/ordering.npy (float64), so
            that two builds can be compared output for output: the inputs are seeded, the same on every run.

N>1: one process per GPU, ONE job (fixed total work -> "strong" scaling at every N): the selection
scan (the Theta(n^3) part) is sharded across the ranks, the per-rank (Q,i,j) partial min-locs are
exchanged through peer-mapped mailboxes over NVLink inside the kernels, the Theta(n^2) update is
replicated (DESIGN.md section 6).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "neighbornet_canonical_order_algorithmic_hbm_throughput"
UNIT = "GB/s"
SCALING = "strong"   # one fixed job at every N


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def sha(o):
    return hashlib.sha256(o.tobytes()).hexdigest()[:16]


def cpu_reference_run(n, seed, threads, want_order=False):
    """One canonical ordering on the CPU restatement; returns (seconds, algorithmic bytes[, ordering])."""
    import oracle
    from fastneighbornet_b200 import synth
    D = synth.additive_noise_matrix(n, seed, 0.05)
    t0 = time.perf_counter()
    o, _, info = oracle.order(D, mode="canonical", want_trace=False, threads=threads)
    dt = time.perf_counter() - t0
    return (dt, info["alg_bytes"], o) if want_order else (dt, info["alg_bytes"])


def dump_outputs(directory, **arrays):
    """--dump-outputs: each array as float64 DIR/<name>.npy (an int32 ordering is exact in float64; n+1 entries stay far
    below 64 MB at any n whose matrix fits a GPU)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), np.asarray(a, dtype=np.float64))


def cubic_fit(ns, ts):
    """least-squares c in t = c*n^3 (BASELINE.md section 4.3)"""
    num = sum(t * n ** 3 for n, t in zip(ns, ts))
    den = sum(float(n) ** 6 for n in ns)
    return num / den


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        self.f.close()
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            sm.sort()
            out["sm_mhz"] = sm[len(sm) // 2]
            out["sm_max_mhz"] = max(mx)
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        return out


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


WORKLOAD = ("canonical Neighbor-Net ordering (-mode Canonical -order), n={n} taxa, synthetic additive tree + 5% noise "
            "(BASELINE metric 'n=20k'; fits one GPU: {gb:.1f} GB fp64 matrix)")


def workload_config(args, world):
    return {
        "workload": WORKLOAD.format(n=args.n, gb=args.n * args.n * 8 / 1e9),
        "n_taxa": args.n, "mode": "canonical", "eps": 0.05,
        "parallelism": "single GPU" if world == 1 else f"{world} GPUs: scan sharded by tile, P2P min-loc mailbox exchange, replicated update",
        "l2": f"input matrix {args.n * args.n * 8 / 1e6:.0f} MB >> 126 MB L2; no explicit flush",
    }


def run_reference(args, rank, world, emit=None):
    """--impl reference: the reference's own CPU algorithm (restatement; the JAR needs a JVM that this image does not have).
    Each step = one canonical ordering of a BOUNDED SAMPLE (n = --ref-n) of the workload with all host threads
    (NeighborNetCanonical's thread partition, NeighborNetCanonical.java:180-206); rank 0 only.  The line says which n it ran
    (`config.n_taxa`), adds the `-threads 1` arm, and fits t = c*n^3 on n in --fit-n to extrapolate the CPU wall time to the
    workload's n (flagged `extrapolated`)."""
    if rank != 0:
        return
    threads = host_threads()
    n = args.ref_n
    for i in range(args.warmup):
        cpu_reference_run(n, 100 + i, threads)
    tot_t, tot_b = 0.0, 0.0
    for i in range(args.steps):
        dt, b, o = cpu_reference_run(n, 1 + i, threads, want_order=True)
        tot_t += dt
        tot_b += b
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ordering=o)
    val = tot_b / tot_t / 1e9
    ms = 1e3 * tot_t / args.steps
    # c*n^3 fits (BASELINE.md section 4.3): all threads on --fit-n, 1 thread on --fit-n1
    fit_ns = [int(x) for x in args.fit_n.split(",") if x]
    fit_ts = []
    for fn_ in fit_ns:
        fit_ts.append(ms / 1e3 if fn_ == n else cpu_reference_run(fn_, 1, threads)[0])
    c_mt = cubic_fit(fit_ns, fit_ts)
    fit1_ns = [int(x) for x in args.fit_n1.split(",") if x]
    fit1 = [cpu_reference_run(fn_, 1, 1) for fn_ in fit1_ns]
    c_1t = cubic_fit(fit1_ns, [t for t, _ in fit1])
    n1 = fit1_ns[-1]
    val1 = fit1[-1][1] / fit1[-1][0] / 1e9
    sample = (f"canonical ordering of a bounded sample, n={n} of the n={args.n} workload (same generator, eps=0.05), {threads} threads, "
              f"NeighborNetCanonical thread partition")
    cfg = workload_config(args, 1)
    cfg.update({"n_taxa": n, "sample_of_n_taxa": args.n, "parallelism": f"CPU, {threads} threads",
                "l2": f"host caches; sample matrix {n * n * 8 / 1e6:.0f} MB"})
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": SCALING,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "value_1thread": val1, "sample_1thread": f"n={n1}, {fit1[-1][0]:.1f} s on 1 thread"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "extrapolated": {
            "extrapolated": True, "n_taxa": args.n, "model": "t = c*n^3 (least squares)",
            "threads_all": {"cores": threads, "fit_n": fit_ns, "fit_seconds": fit_ts, "c": c_mt, "seconds_at_workload_n": c_mt * args.n ** 3,
                            "seconds_at_100k": c_mt * 1e15},
            "threads_1": {"cores": 1, "fit_n": fit1_ns, "fit_seconds": [t for t, _ in fit1], "c": c_1t,
                          "seconds_at_workload_n": c_1t * args.n ** 3, "seconds_at_100k": c_1t * 1e15},
        },
    }
    (emit or (lambda l: print(json.dumps(l), flush=True)))(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=20000)
    ap.add_argument("--ref-n", type=int, default=2000, help="taxa of the bounded CPU sample")
    ap.add_argument("--fit-n", default="2000,5000,10000", help="reference arm: sizes of the all-threads c*n^3 fit")
    ap.add_argument("--fit-n1", default="1000,1500,2000", help="reference arm: sizes of the 1-thread c*n^3 fit")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--csw-n", type=int, default=400, help="taxa of the split-weight config entry")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's ordering to DIR/ordering.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    # stdout carries exactly ONE JSON line: libraries that print there (NCCL's version banner) are sent to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        os.write(json_fd, (json.dumps(line) + "\n").encode())

    if args.impl == "reference":
        run_reference(args, rank, world, emit)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import fastneighbornet_b200 as fnn
    from fastneighbornet_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"   # keep stdout to the one JSON line (NCCL prints its version banner there)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_hashes(h):
        if world == 1:
            return [h]
        hs = [None] * world
        dist.all_gather_object(hs, h)
        return hs

    # ---- parity at THIS world size, before anything is timed (VERDICT r1 "next" 1a)
    parity = None
    if not args.no_parity:
        import oracle
        parity = {"world": world, "ok": True, "cases": []}
        for pn, pseed in ((1500, 7), (5000, 3)):
            D = synth.additive_noise_matrix(pn, pseed, 0.05)
            with fnn.Context(pn, device=local_rank, record_trace=1) as pc:
                if world > 1:
                    pc.connect_torch()
                pc.load_host(D)
                po = pc.order()
                ptr = pc.trace()
            hs = gather_hashes(sha(po))
            case = {"n": pn, "ordering_sha256": hs[0], "ranks_agree": len(set(hs)) == 1}
            if rank == 0:
                o_ref, tr_ref, _ = oracle.order(D, threads=host_threads())
                case["ordering_equals_oracle"] = bool((po == o_ref).all())
                case["trace_equals_oracle"] = bool(ptr.shape == tr_ref.shape and (ptr == tr_ref).all())
                case["oracle_sha256"] = sha(o_ref)
                parity["ok"] = parity["ok"] and case["ordering_equals_oracle"] and case["trace_equals_oracle"] and case["ranks_agree"]
            parity["cases"].append(case)
            del D
        barrier()

    n = args.n
    seed = 1   # every rank holds the same matrix (one job)
    ctx = fnn.Context(n, device=local_rank, use_graph=1)
    if world > 1:
        ctx.connect_torch()
    # pristine device copy of the input (torch owns it: plumbing, not the product)
    ctx.synth(seed, 0.05)
    dptr, ld = ctx.matrix_ptr()
    pristine = torch.empty((n, ld), dtype=torch.float64, device=f"cuda:{local_rank}")
    # view of the library's device matrix through __cuda_array_interface__ (zero copy)

    class _View:
        def __init__(self, ptr, shape):
            self.__cuda_array_interface__ = {"shape": shape, "typestr": "<f8", "data": (ptr, False), "version": 3}

    view = torch.as_tensor(_View(dptr, (n, ld)), device=f"cuda:{local_rank}")
    pristine.copy_(view)
    torch.cuda.synchronize()

    # N>1: the hash an un-wired single-GPU run of the same workload gives (rank 0), for the driver to compare across N
    sha_n1 = None
    if world > 1 and not args.no_parity:
        if rank == 0:
            with fnn.Context(n, device=local_rank, use_graph=1) as c1:
                c1.load_device(pristine.data_ptr(), ld)
                sha_n1 = sha(c1.order())
        barrier()

    def step():
        ctx.load_device(pristine.data_ptr(), ld)
        return ctx.order()

    ordering0 = None
    for _ in range(args.warmup):
        ordering0 = step()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    t0 = time.perf_counter()
    dev_ms, launches, alg_bytes = 0.0, 0, 0.0
    o = ordering0
    for _ in range(args.steps):
        o = step()
        st = ctx.stats()
        dev_ms += st["order_ms"]
        launches += st["kernel_launches"]
        alg_bytes += st["scan_alg_bytes"]
    barrier()
    elapsed = time.perf_counter() - t0
    clocks = sampler.stop() if sampler else None
    if ordering0 is not None:
        assert (o == ordering0).all(), "ordering changed between identical steps"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ordering=o)
    picks = (st["picks_certified"], st["picks_exact"])
    # max over ranks of the elapsed time; launches summed over ranks
    if world > 1:
        t = torch.tensor([elapsed, dev_ms], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed, dev_ms = float(t[0]), float(t[1])
        b = torch.tensor([float(launches)], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(b, op=dist.ReduceOp.SUM)
        launches = int(b[0])   # alg_bytes is the ONE job's (identical on every rank)
    value = alg_bytes / elapsed / 1e9
    hashes = gather_hashes(sha(o))
    if parity is not None:
        parity["workload_ranks_agree"] = len(set(hashes)) == 1
        parity["ok"] = parity["ok"] and parity["workload_ranks_agree"]
        if sha_n1 is not None:
            parity["workload_equals_single_gpu"] = (hashes[0] == sha_n1)
            parity["ok"] = parity["ok"] and parity["workload_equals_single_gpu"]

    # ---- e2e: one-shot C-ABI call with a pinned HOST matrix
    e2e = None
    if not args.no_e2e:
        host = torch.empty((n, n), dtype=torch.float64).pin_memory()
        host.copy_(pristine[:, :n])  # the ctx matrix itself was consumed by the runs above
        torch.cuda.synchronize()
        Dh = host.numpy()

        def e2e_step():
            if world == 1:
                return fnn.order(Dh, device=local_rank)   # the one-shot reference-facing seam (fnn_order)
            ctx.load_host_sharded(Dh)                     # N>1: each rank uploads 1/world of the rows, NVLink does the rest
            return ctx.order()

        if world == 1:
            ctx.close()
        e2e_step()  # warm-up (allocator, graph instantiation)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            oe = e2e_step()
        barrier()
        e2e_elapsed = time.perf_counter() - t0
        assert (oe == o).all(), "e2e ordering differs from the device-resident run"
        if world > 1:
            t = torch.tensor([e2e_elapsed], dtype=torch.float64, device=f"cuda:{local_rank}")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_elapsed = float(t[0])
        e2e = {"value": alg_bytes / e2e_elapsed / 1e9, "unit": UNIT, "h2d_bytes_per_step": n * n * 8,   # N>1: 1/world of the rows per rank over PCIe, the rest over NVLink
               "d2h_bytes_per_step": (n + 1) * 4 * world, "ms_per_step": 1e3 * e2e_elapsed / args.steps}
        if world == 1:
            fnn.release_cache()
        del host, Dh

    # ---- roofline of the dominant kernel (k_scan_tma), rank 0 only
    roofline, cpu_baseline, configs = None, None, None
    peak, peak_src = measured_peak()
    if rank == 0:
        pctx = fnn.Context(n, device=local_rank, profile_every=16)
        pctx.load_device(pristine.data_ptr(), ld)
        pctx.order()
        ps = pctx.stats()
        pctx.close()
        achieved = ps["prof_scan_bytes"] / (ps["prof_scan_ms"] * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": "k_scan_tma", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "frac_of_nominal_8000": achieved / 8000.0,
                    "traffic": None, "peak_source": peak_src, "samples": ps["prof_scan_samples"],
                    "avg_launch_ms": ps["prof_scan_ms"] / max(1, ps["prof_scan_samples"]),
                    "alg_bytes_per_launch": ps["prof_scan_bytes"] / max(1, ps["prof_scan_samples"]),
                    "scan_share_of_step": ((ps["prof_scan_ms"] * 16) / (1e3 * elapsed / args.steps)) if world == 1 else None,
                    "whole_job_frac": value / (peak * world)}
        if world > 1:
            roofline["note"] = "kernel profiled on rank 0 as a single-GPU run of the same workload (each rank launches it on 1/world of the tiles)"
        tfile = os.path.join(ROOT, "profiles", "scan_traffic.json")
        if os.path.exists(tfile):
            try:
                with open(tfile) as f:
                    tj = json.load(f)
                roofline["traffic"] = tj.get("traffic_bytes_per_launch")
                # the ncu capture is of the first launches (m ~ n): compare it with THAT launch's algorithmic bytes
                roofline["traffic_launch_alg_bytes"] = tj.get("alg_bytes_same_launch")
                roofline["traffic_source"] = tj.get("source")
            except Exception:
                pass
    del pristine
    if world == 1:
        try:
            ctx.close()
        except Exception:
            pass
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs that fit the step budget, one timed run each (N=1 only)
    if rank == 0 and world == 1 and not args.no_configs:
        configs = []

        def timed(label, cn, cseed, eps, unit_bytes_key, **opts):
            with fnn.Context(cn, device=local_rank, **opts) as c:
                c.synth(cseed, eps)
                c.order()           # warm-up (graph instantiation, clocks)
                c.synth(cseed, eps)
                torch.cuda.synchronize()
                t0_ = time.perf_counter()
                oo = c.order()
                dt = time.perf_counter() - t0_
                s_ = c.stats()
            b_ = s_[unit_bytes_key] + (s_["scan_alg_bytes"] if unit_bytes_key != "scan_alg_bytes" else 0.0)
            return {"config": label, "n_taxa": cn, "ms": 1e3 * dt, "alg_bytes": b_, "achieved": b_ / dt / 1e9, "unit": "GB/s",
                    "frac": b_ / dt / 1e9 / peak, "iterations": s_["iterations"], "gpu_launches": s_["kernel_launches"],
                    "strategy_units": s_["strategy_units"], "ordering_sha256": sha(oo)}

        configs.append(timed("configs[0]: Canonical -order, 200-taxon additive tree (eps=0)", 200, 1, 0.0, "scan_alg_bytes"))
        configs.append(timed("configs[1] ordering stage: Canonical, 5000 taxa", 5000, 2, 0.05, "scan_alg_bytes"))
        # configs[1] split-weight stage (CircularSplitWeights active-set + CG) at the size that fits the step budget; the roofline of
        # ONE CG iteration is SURVEY 8(d)'s 112 * npairs algorithmic bytes / measured time per iteration
        csn = args.csw_n
        Dc = synth.additive_noise_matrix(csn, 1, 0.05)
        oc = fnn.order(Dc, device=local_rank)
        duc = synth.upper_triangle(Dc)
        fnn.split_weights(oc, duc, constrained=False, device=local_rank)   # warm-up
        t0_ = time.perf_counter()
        xc, stc = fnn.split_weights(oc, duc, device=local_rank)
        dtc = time.perf_counter() - t0_
        npairs = csn * (csn - 1) // 2
        us_it = 1e6 * dtc / max(1, stc["cg_iters"])
        configs.append({"config": f"configs[1] split-weight stage at the size that fits the step budget: CircularSplitWeights (active set + CG), {csn} taxa",
                        "n_taxa": csn, "ms": 1e3 * dtc, "cg_iterations": stc["cg_iters"], "cg_solves": stc["cg_calls"], "us_per_cg_iteration": us_it,
                        "alg_bytes_per_cg_iteration": 112.0 * npairs, "achieved": 112.0 * npairs / (us_it * 1e-6) / 1e9, "unit": "GB/s",
                        "frac": 112.0 * npairs / (us_it * 1e-6) / 1e9 / peak, "gpu_launches": stc["kernel_launches"], "kept_splits": int((xc > 1e-6).sum()),
                        "bound": "barrier/L2 latency at this size (8 grid barriers per iteration, DESIGN.md 4.3), HBM only above n ~ 3000"})
        # the full-size configs[1] run (5000 taxa: 52 minutes) does not fit a bench step; its committed record rides along
        full = os.path.join(ROOT, "profiles", "r2_config1_n5000.json")
        if os.path.exists(full):
            try:
                with open(full) as f_:
                    configs[-1]["full_size_builder_run"] = dict(json.load(f_), source="profiles/r2_config1_n5000.json (tools/config1_run.py 5000, not re-run here)")
            except Exception:
                pass
        fnn.release_cache()
        configs.append(timed("configs[2] without -additive: Relaxed, 20000 taxa (row scans: SURVEY 8d K7 bytes + the canonical tail's scan bytes)",
                             20000, 3, 0.05, "strategy_alg_bytes", mode="relaxed", seed=7))
        configs.append(timed("configs[3] at the size that fits the step budget: Random_NLOGN -mult 5, 10000 taxa (samples: SURVEY 8d K9 bytes + tail scan bytes)",
                             10000, 4, 0.05, "strategy_alg_bytes", mode="random_nlogn", mult=5, seed=7))

    if rank == 0 and not args.no_cpu_baseline and world == 1:   # reported at N=1 only
        threads = host_threads()
        dt, b = cpu_reference_run(args.ref_n, 1, threads)
        cpu_baseline = {"value": b / dt / 1e9, "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": f"one canonical ordering at n={args.ref_n} (bounded sample of the n={n} workload, same generator), "
                                  f"{dt:.1f} s on {threads} threads"}
        n1 = min(args.ref_n, 1500)   # the reference's -threads 1 figure on a smaller sample (SURVEY section 8d)
        dt1, b1 = cpu_reference_run(n1, 1, 1)
        cpu_baseline["value_1thread"] = b1 / dt1 / 1e9
        cpu_baseline["sample_1thread"] = f"n={n1}, {dt1:.1f} s on 1 thread"
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * elapsed / args.steps, "higher_is_better": True, "scaling": SCALING, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": workload_config(args, world),
        "device_ms_per_step": dev_ms / args.steps, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
        "ordering_sha256": hashes[0], "ordering_sha256_single_gpu": sha_n1 if world > 1 else hashes[0], "parity": parity,
        "picks": {"certified": picks[0], "exact_sums": picks[1]},
        "roofline": roofline, "cpu_baseline": cpu_baseline, "configs": configs,
    }
    emit(line)


if __name__ == "__main__":
    main()
