"""ctypes binding of libfastnn.so plus classes that mirror the reference's operator API.

Reference interface mirrored (argument meaning and error behaviour kept):
  new NeighborNetCanonical(double[][] D, int nTaxa, int nThreads, ExecutorService pool)
  new NeighborNetLocal(D, nTaxa, nThreads, boolean additive, pool)
  new NeighborNetRandom(D, nTaxa, nThreads, pool, RandomAmount amount, int mult)
  int[] runNeighborNet()                                   (NetMakerOriginal.java:51,129)
`nThreads`/`pool` are accepted and ignored (single host control thread; SURVEY §8b).
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class FastNNError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libfastnn error {code}: {msg}")
        self.code = code


class fnn_opts(ctypes.Structure):
    _fields_ = [
        ("mode", ctypes.c_int32),
        ("mult", ctypes.c_int32),
        ("additive", ctypes.c_int32),
        ("canonical_fallback", ctypes.c_int32),
        ("seed", ctypes.c_int64),
        ("device", ctypes.c_int32),
        ("use_graph", ctypes.c_int32),
        ("record_trace", ctypes.c_int32),
        ("profile_every", ctypes.c_int32),
        ("reserved", ctypes.c_int32 * 6),
    ]


class fnn_stats(ctypes.Structure):
    _fields_ = [
        ("iterations", ctypes.c_int64),
        ("kernel_launches", ctypes.c_int64),
        ("scan_launches", ctypes.c_int64),
        ("scan_alg_bytes", ctypes.c_double),
        ("prof_scan_ms", ctypes.c_double),
        ("prof_scan_bytes", ctypes.c_double),
        ("prof_scan_samples", ctypes.c_int64),
        ("order_ms", ctypes.c_double),
        ("h2d_ms", ctypes.c_double),
        ("reserved", ctypes.c_double * 8),
    ]


MODES = {"canonical": 0, "relaxed": 1, "random_n": 2, "random_nlogn": 3, "random_logn": 4}

# every symbol include/fastnn.h declares (checked by tests/test_abi.py)
ABI_SYMBOLS = [
    "fnn_default_opts", "fnn_last_error", "fnn_device_count", "fnn_ctx_create", "fnn_ctx_destroy",
    "fnn_ctx_load_host", "fnn_ctx_load_device", "fnn_ctx_synth", "fnn_ctx_read_matrix", "fnn_ctx_order",
    "fnn_ctx_trace", "fnn_ctx_stats", "fnn_ctx_matrix_ptr", "fnn_order", "fnn_rowsums", "fnn_seq_sum",
    "fnn_split_weights", "fnn_csw_matvec", "fnn_ctx_ipc_handle", "fnn_ctx_connect", "fnn_weighted_splits", "fnn_network",
    "fnn_phylip_taxa", "fnn_read_phylip", "fnn_write_nexus", "fnn_java_double_to_string", "fnn_release_cache",
    "fnn_ctx_load_host_rows", "fnn_ctx_commit_load", "fnn_split_weights_budget", "fnn_ctx_strategy_record",
    "fnn_ctx_prune_bounds", "fnn_alignment_size", "fnn_read_alignment", "fnn_ctx_load_alignment", "fnn_distances",
]

# enum fnn_dist_model: distances from a nucleotide alignment (include/fastnn.h)
MODELS = {"p": 0, "jc69": 1, "k2p": 2}


def lib_path():
    # FNN_LIB: an alternative build of the same library (e.g. one compiled with -DFNN_XSUM_TIMING for a profiling session)
    return os.environ.get("FNN_LIB") or os.path.join(_HERE, "libfastnn.so")


def lib():
    """Load libfastnn.so; fails loudly when the CUDA extension has not been built."""
    global _LIB
    if _LIB is None:
        p = lib_path()
        if not os.path.exists(p):
            raise FastNNError(-100, f"{p} is missing: run ./build.sh (nvcc, sm_100a). There is no CPU fallback.")
        L = ctypes.CDLL(p)
        vp, c_dp = ctypes.c_void_p, ctypes.POINTER(ctypes.c_double)
        L.fnn_default_opts.argtypes = [ctypes.POINTER(fnn_opts)]
        L.fnn_default_opts.restype = None
        L.fnn_last_error.restype = ctypes.c_char_p
        L.fnn_device_count.restype = ctypes.c_int
        L.fnn_ctx_create.argtypes = [ctypes.POINTER(fnn_opts), ctypes.c_int64, ctypes.POINTER(vp)]
        L.fnn_ctx_destroy.argtypes = [vp]
        L.fnn_ctx_destroy.restype = None
        L.fnn_ctx_load_host.argtypes = [vp, c_dp]
        L.fnn_ctx_load_device.argtypes = [vp, vp, ctypes.c_int64]
        L.fnn_ctx_load_host_rows.argtypes = [vp, c_dp, ctypes.c_int64, ctypes.c_int64]
        L.fnn_ctx_commit_load.argtypes = [vp]
        L.fnn_ctx_synth.argtypes = [vp, c_dp, c_dp, ctypes.POINTER(ctypes.c_int64), ctypes.c_uint64, ctypes.c_double]
        L.fnn_ctx_read_matrix.argtypes = [vp, c_dp]
        L.fnn_ctx_order.argtypes = [vp, ctypes.POINTER(ctypes.c_int32)]
        L.fnn_ctx_trace.argtypes = [vp, c_dp, ctypes.c_int64]
        L.fnn_ctx_trace.restype = ctypes.c_int64
        L.fnn_ctx_strategy_record.argtypes = [vp, ctypes.POINTER(ctypes.c_int64), ctypes.c_int64]
        L.fnn_ctx_prune_bounds.argtypes = [vp, ctypes.c_int64, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                           ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_double),
                                           ctypes.POINTER(ctypes.c_int64)]
        L.fnn_ctx_strategy_record.restype = ctypes.c_int64
        L.fnn_ctx_stats.argtypes = [vp, ctypes.POINTER(fnn_stats)]
        L.fnn_ctx_matrix_ptr.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_int64)]
        L.fnn_ctx_ipc_handle.argtypes = [vp, ctypes.c_char_p]
        L.fnn_ctx_connect.argtypes = [vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_char_p]
        L.fnn_order.argtypes = [ctypes.POINTER(fnn_opts), c_dp, ctypes.c_char_p, ctypes.c_int64, ctypes.POINTER(ctypes.c_int32)]
        L.fnn_release_cache.argtypes = []
        L.fnn_release_cache.restype = None
        L.fnn_rowsums.argtypes = [ctypes.POINTER(fnn_opts), c_dp, ctypes.c_int64, c_dp]
        L.fnn_split_weights.argtypes = [ctypes.POINTER(fnn_opts), ctypes.POINTER(ctypes.c_int32), c_dp, ctypes.c_int64, c_dp,
                                        ctypes.POINTER(ctypes.c_int64)]
        L.fnn_split_weights_budget.argtypes = [ctypes.POINTER(fnn_opts), ctypes.POINTER(ctypes.c_int32), c_dp, ctypes.c_int64,
                                               ctypes.c_int64, ctypes.c_int64, c_dp, ctypes.POINTER(ctypes.c_uint8),
                                               ctypes.POINTER(ctypes.c_int64)]
        L.fnn_weighted_splits.argtypes = [ctypes.POINTER(fnn_opts), ctypes.POINTER(ctypes.c_int32), c_dp, ctypes.c_int64, ctypes.c_double,
                                          ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32), c_dp, ctypes.c_int64,
                                          ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]
        L.fnn_phylip_taxa.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_int64)]
        L.fnn_read_phylip.argtypes = [ctypes.c_char_p, ctypes.c_int64, c_dp, ctypes.c_char_p, ctypes.c_int64, ctypes.c_int]
        ip32 = ctypes.POINTER(ctypes.c_int32)
        L.fnn_write_nexus.argtypes = [ctypes.c_char_p, ctypes.c_int64, ctypes.c_char_p, ctypes.c_int64, c_dp, ip32, ip32, ip32, c_dp,
                                      ctypes.c_int64, ctypes.c_int]
        L.fnn_java_double_to_string.argtypes = [ctypes.c_double, ctypes.c_char_p, ctypes.c_int64]
        L.fnn_network.argtypes = [ctypes.POINTER(fnn_opts), c_dp, ctypes.c_int64, ctypes.c_double, ctypes.POINTER(ctypes.c_int32),
                                  ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32), c_dp, ctypes.c_int64,
                                  ctypes.POINTER(ctypes.c_int64)]
        L.fnn_csw_matvec.argtypes = [ctypes.POINTER(fnn_opts), ctypes.c_int32, c_dp, ctypes.c_int64, c_dp]
        L.fnn_seq_sum.argtypes = [ctypes.POINTER(fnn_opts), c_dp, ctypes.c_int32, ctypes.c_int64, c_dp]
        c_bp = ctypes.POINTER(ctypes.c_uint8)
        L.fnn_alignment_size.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]
        L.fnn_read_alignment.argtypes = [ctypes.c_char_p, ctypes.c_int64, ctypes.c_int64, c_bp, ctypes.c_char_p, ctypes.c_int64,
                                         ctypes.c_int]
        L.fnn_ctx_load_alignment.argtypes = [vp, c_bp, ctypes.c_int64, ctypes.c_int32, ctypes.c_double]
        L.fnn_distances.argtypes = [ctypes.POINTER(fnn_opts), c_bp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.c_double,
                                    c_dp]
        _LIB = L
    return _LIB


def _check(rc):
    if rc != 0:
        raise FastNNError(rc, lib().fnn_last_error().decode())


def device_count():
    return lib().fnn_device_count()


# A/B switches carried in fnn_opts.reserved (include/fastnn.h): name -> (index, bit or None for "whole int")
_RESERVED = {"no_prune": (0, None), "serial_chain": (1, None), "no_overlap": (5, 1), "force_exact_pick": (5, 2), "csw_variant": (4, None)}
CSW_VARIANTS = {"default": 0, "graph": 1, "literal": 2}


def default_opts(**kw):
    o = fnn_opts()
    lib().fnn_default_opts(ctypes.byref(o))
    for k, v in kw.items():
        if k == "mode" and isinstance(v, str):
            v = MODES[v.lower()]
        if k in _RESERVED:
            idx, bit = _RESERVED[k]
            if bit is None:
                o.reserved[idx] = int(v)
            elif v:
                o.reserved[idx] |= bit
            continue
        setattr(o, k, int(v))
    return o


def _dp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def _alignment_args(codes, model, undefined):
    """codes as a C-contiguous uint8 [n, L] array, the model's enum value and undefined_value (None -> NaN: fail)."""
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    if codes.ndim != 2:
        raise ValueError("codes must be a 2-D [taxa, sites] array")
    if model not in MODELS:
        raise ValueError(f"model must be one of {', '.join(MODELS)}")
    return codes, MODELS[model], float("nan") if undefined is None else float(undefined)


class Context:
    """Device-resident problem of n taxa (fnn_ctx)."""

    def __init__(self, n, **opts):
        self.n = int(n)
        self.opts = default_opts(**opts)
        self._h = ctypes.c_void_p()
        _check(lib().fnn_ctx_create(ctypes.byref(self.opts), self.n, ctypes.byref(self._h)))

    def close(self):
        if self._h:
            lib().fnn_ctx_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def load_host(self, D):
        D = np.ascontiguousarray(D, dtype=np.float64)
        assert D.shape == (self.n, self.n)
        _check(lib().fnn_ctx_load_host(self._h, _dp(D)))

    def load_host_rows(self, D_rows, row0):
        """Upload rows [row0, row0 + len(D_rows)) only (fnn_ctx_load_host_rows); finish with commit_load()."""
        D_rows = np.ascontiguousarray(D_rows, dtype=np.float64)
        assert D_rows.ndim == 2 and D_rows.shape[1] == self.n
        _check(lib().fnn_ctx_load_host_rows(self._h, _dp(D_rows), int(row0), D_rows.shape[0]))

    def commit_load(self):
        _check(lib().fnn_ctx_commit_load(self._h))

    def load_host_sharded(self, D):
        """N>1 (torch.distributed initialised, contexts wired): every rank uploads 1/world of the rows over its own PCIe
        link, the row blocks then travel between the GPUs over NVLink (NCCL broadcast on the library's device matrix) -
        n*n*8 bytes cross PCIe in total instead of n*n*8 per rank."""
        import torch
        import torch.distributed as dist
        D = np.ascontiguousarray(D, dtype=np.float64)
        assert D.shape == (self.n, self.n)
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return self.load_host(D)
        world, rank = dist.get_world_size(), dist.get_rank()
        bounds = [self.n * r // world for r in range(world + 1)]
        r0, r1 = bounds[rank], bounds[rank + 1]
        _check(lib().fnn_ctx_load_host_rows(self._h, _dp(D[r0:r1]), r0, r1 - r0))
        dptr, ld = self.matrix_ptr()

        class _View:
            def __init__(s_, ptr, shape):
                s_.__cuda_array_interface__ = {"shape": shape, "typestr": "<f8", "data": (ptr, False), "version": 3}

        dev = torch.device("cuda", int(self.opts.device))
        view = torch.as_tensor(_View(dptr, (self.n, ld)), device=dev)
        for r in range(world):
            if bounds[r + 1] > bounds[r]:
                dist.broadcast(view[bounds[r]:bounds[r + 1]], src=r)
        torch.cuda.synchronize(dev)
        _check(lib().fnn_ctx_commit_load(self._h))

    def load_device(self, dptr, ld):
        _check(lib().fnn_ctx_load_device(self._h, ctypes.c_void_p(int(dptr)), int(ld)))

    def synth(self, seed, eps=0.05):
        from . import synth as _s
        h, a, pi, inv = _s.tree_params(self.n, seed)
        h = np.ascontiguousarray(h, dtype=np.float64)
        a = np.ascontiguousarray(a, dtype=np.float64)
        inv = np.ascontiguousarray(inv, dtype=np.int64)
        if h.size == 0:
            h = np.zeros(1)
        _check(lib().fnn_ctx_synth(self._h, _dp(h), _dp(a), inv.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
                                   ctypes.c_uint64(_s.stream_base(seed, 3)), float(eps)))

    def load_alignment(self, codes, model="p", undefined=None):
        """Distances of an [n, L] code array (read_alignment) computed on the device into this context's matrix
        (fnn_ctx_load_alignment).  undefined=None: an undefined pair is an error; a finite value >= 0 is stored there."""
        codes, m, u = _alignment_args(codes, model, undefined)
        assert codes.shape[0] == self.n
        _check(lib().fnn_ctx_load_alignment(self._h, codes.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), codes.shape[1], m, u))

    def read_matrix(self):
        out = np.empty((self.n, self.n), dtype=np.float64)
        _check(lib().fnn_ctx_read_matrix(self._h, _dp(out)))
        return out

    def matrix_ptr(self):
        p, ld = ctypes.c_void_p(), ctypes.c_int64()
        _check(lib().fnn_ctx_matrix_ptr(self._h, ctypes.byref(p), ctypes.byref(ld)))
        return p.value, ld.value

    def ipc_handle(self):
        buf = ctypes.create_string_buffer(64)
        _check(lib().fnn_ctx_ipc_handle(self._h, buf))
        return buf.raw

    def connect(self, rank, world, handles):
        """handles: list of the `world` 64-byte IPC handles in rank order (e.g. from all_gather_object)."""
        assert len(handles) == world and all(len(h) == 64 for h in handles)
        _check(lib().fnn_ctx_connect(self._h, int(rank), int(world), b"".join(handles)))

    def connect_torch(self):
        """Wire the ranks of the default torch.distributed group (one process per GPU)."""
        import torch.distributed as dist
        world, rank = dist.get_world_size(), dist.get_rank()
        handles = [None] * world
        dist.all_gather_object(handles, self.ipc_handle())
        self.connect(rank, world, handles)
        dist.barrier()

    def order(self):
        out = np.zeros(self.n + 1, dtype=np.int32)
        _check(lib().fnn_ctx_order(self._h, out.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))))
        return out

    def trace(self):
        rows = np.zeros((self.n + 8, 8), dtype=np.float64)
        k = lib().fnn_ctx_trace(self._h, _dp(rows), rows.shape[0])
        if k < 0:
            _check(int(k))
        return rows[: int(k)]

    def strategy_record(self):
        """Per-iteration strategy record (fnn_ctx_strategy_record; needs record_trace=1): an (iterations, 4) int64 array,
        Random: draws, rejected draws, remapped draws, digest; Relaxed: row scans, ties, look-aheads, digest.  Column 3 is a
        uint64 digest stored as int64 (view it with .view(np.uint64))."""
        rows = np.zeros((self.n + 8, 4), dtype=np.int64)
        k = lib().fnn_ctx_strategy_record(self._h, rows.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), rows.shape[0])
        if k < 0:
            _check(int(k))
        return rows[: int(k)]

    def prune_bounds(self, iters):
        """State of the scan's pruning bounds after the first `iters` iterations (fnn_ctx_prune_bounds; consumes the loaded
        matrix): dict with D (slot layout), segmin (n, S), smax (S,) decoded to float64 (NaN = none), Sx, m, P2, mask_su,
        iter, done."""
        n = self.n
        S = (((n + 15) // 16 * 16) + 255) // 256
        D = np.empty((n, n)); segmin = np.empty((n, S)); sx = np.empty(n)
        keys = np.zeros(S, dtype=np.uint64); meta = np.zeros(6, dtype=np.int64)
        _check(lib().fnn_ctx_prune_bounds(self._h, int(iters), _dp(D), _dp(segmin),
                                          keys.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), _dp(sx),
                                          meta.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))))
        assert int(meta[4]) == S
        top = (keys >> np.uint64(63)).astype(bool)
        bits = np.where(top, keys & np.uint64(0x7FFFFFFFFFFFFFFF), ~keys)
        smax = bits.view(np.float64).copy()
        smax[keys == 0] = np.nan
        return {"D": D, "segmin": segmin, "smax": smax, "Sx": sx, "m": int(meta[0]), "P2": int(meta[1]),
                "mask_su": int(meta[2]), "iter": int(meta[3]), "done": int(meta[5])}

    def stats(self):
        s = fnn_stats()
        _check(lib().fnn_ctx_stats(self._h, ctypes.byref(s)))
        out = {f: getattr(s, f) for f, _ in fnn_stats._fields_ if f != "reserved"}
        out["picks_certified"] = int(s.reserved[0])   # 4-candidate picks decided by the bounded parallel ComputeRx sums
        out["picks_exact"] = int(s.reserved[1])       # ... that needed the exact left-to-right sums
        out["strategy_alg_bytes"] = float(s.reserved[2])   # Relaxed row scans / Random samples (SURVEY 8d K7/K9)
        out["strategy_units"] = int(s.reserved[3])
        out["scan_read_bytes"] = float(s.reserved[4])      # matrix bytes the selection scan fetched (pruned segments not)
        out["scan_units_skipped"] = int(s.reserved[5])     # row segments the pruned scans did not fetch
        out["dist_pack_ms"] = float(s.reserved[6])         # load_alignment: bit-plane packing kernel (h2d_ms: the codes' upload)
        out["dist_pairs_ms"] = float(s.reserved[7])        # load_alignment: pair kernel
        return out


def order(D=None, phylip_path=None, n=None, **opts):
    """One-shot seam B1 (fnn_order): host matrix or Phylip path in, ordering[n+1] out."""
    o = default_opts(**opts)
    if D is not None:
        D = np.ascontiguousarray(D, dtype=np.float64)
        n = D.shape[0]
    out = np.zeros(int(n) + 1, dtype=np.int32)
    _check(lib().fnn_order(ctypes.byref(o), _dp(D) if D is not None else None,
                           phylip_path.encode() if phylip_path else None, int(n),
                           out.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))))
    return out


def release_cache():
    """Free the context the one-shot seam keeps between calls (fnn_release_cache)."""
    lib().fnn_release_cache()


def rowsums(D, **opts):
    D = np.ascontiguousarray(D, dtype=np.float64)
    o = default_opts(**opts)
    out = np.zeros(D.shape[0], dtype=np.float64)
    _check(lib().fnn_rowsums(ctypes.byref(o), _dp(D), D.shape[0], _dp(out)))
    return out


def seq_sum(rows, serial=False, **opts):
    """Left-to-right fp64 sums of up to 4 equally long rows on the device (fnn_seq_sum)."""
    rows = np.ascontiguousarray(np.atleast_2d(rows), dtype=np.float64)
    o = default_opts(**opts)
    o.reserved[1] = 1 if serial else 0
    out = np.zeros(rows.shape[0], dtype=np.float64)
    _check(lib().fnn_seq_sum(ctypes.byref(o), _dp(rows), rows.shape[0], rows.shape[1], _dp(out)))
    return out


def split_weights(ordering, d_upper, constrained=True, variant="default", **opts):
    """Seam B2 (fnn_split_weights): CircularSplitWeights.getWeights(ntax, ordering, d, v="ols", constrained, ...)
    (CircularSplitWeights.java:162).  Returns (x[npairs] in the live split indexing, stats dict).
    variant: "default" (production formulation), "graph" (launch-per-phase A/B path), "literal" (the reference's own
    operation order on the device, n <= 512: the validation mode held bit for bit against the literal oracle)."""
    opts = dict(opts, csw_variant=CSW_VARIANTS[variant])
    ordering = np.ascontiguousarray(ordering, dtype=np.int32)
    n = ordering.shape[0] - 1
    d_upper = np.ascontiguousarray(d_upper, dtype=np.float64)
    assert d_upper.shape[0] == n * (n - 1) // 2
    o = default_opts(**opts)
    o.reserved[3] = 0 if constrained else 1
    x = np.zeros_like(d_upper)
    st = np.zeros(5, dtype=np.int64)
    _check(lib().fnn_split_weights(ctypes.byref(o), ordering.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), _dp(d_upper), n,
                                   _dp(x), st.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))))
    return x, {"cg_iters": int(st[0]), "cg_calls": int(st[1]), "outer": int(st[2]), "inner": int(st[3]), "kernel_launches": int(st[4])}


def split_weights_budget(ordering, d_upper, max_cg_iters=0, max_cg_calls=0, variant="default", **opts):
    """fnn_split_weights_budget: split_weights with every CG call capped at max_cg_iters iterations and the solver stopped
    right after its max_cg_calls-th CG call (0 = no limit; both 0 = split_weights).  For parity tests at production sizes.
    Returns (x[npairs], active[npairs] bool, stats dict as split_weights)."""
    opts = dict(opts, csw_variant=CSW_VARIANTS[variant])
    ordering = np.ascontiguousarray(ordering, dtype=np.int32)
    n = ordering.shape[0] - 1
    d_upper = np.ascontiguousarray(d_upper, dtype=np.float64)
    assert d_upper.shape[0] == n * (n - 1) // 2
    o = default_opts(**opts)
    x = np.zeros_like(d_upper)
    active = np.zeros(d_upper.shape[0], dtype=np.uint8)
    st = np.zeros(5, dtype=np.int64)
    _check(lib().fnn_split_weights_budget(ctypes.byref(o), ordering.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), _dp(d_upper), n,
                                          int(max_cg_iters), int(max_cg_calls), _dp(x),
                                          active.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)),
                                          st.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))))
    return x, active.astype(bool), {"cg_iters": int(st[0]), "cg_calls": int(st[1]), "outer": int(st[2]), "inner": int(st[3]),
                                    "kernel_launches": int(st[4])}


def network_splits(ordering, d_upper, cutoff=1e-6, constrained=True, **opts):
    """fnn_weighted_splits: solve and emit only the kept splits, compacted on the device.
    Returns (split_i, split_j, weight) arrays; split k is the taxon set {ordering[split_i[k]+1 .. split_j[k]]}."""
    ordering = np.ascontiguousarray(ordering, dtype=np.int32)
    n = ordering.shape[0] - 1
    d_upper = np.ascontiguousarray(d_upper, dtype=np.float64)
    o = default_opts(**opts)
    o.reserved[3] = 0 if constrained else 1
    cap = n * (n - 1) // 2
    si, sj, w = np.zeros(cap, dtype=np.int32), np.zeros(cap, dtype=np.int32), np.zeros(cap, dtype=np.float64)
    kept = ctypes.c_int64()
    ip = ctypes.POINTER(ctypes.c_int32)
    _check(lib().fnn_weighted_splits(ctypes.byref(o), ordering.ctypes.data_as(ip), _dp(d_upper), n, float(cutoff),
                                     si.ctypes.data_as(ip), sj.ctypes.data_as(ip), _dp(w), cap, ctypes.byref(kept), None))
    k = kept.value
    return si[:k].copy(), sj[:k].copy(), w[:k].copy()


def read_phylip(path, threads=0, name_len=64):
    """Native Phylip loader (fnn_phylip_taxa + fnn_read_phylip; host only, no device needed).
    Returns (D[n, n] float64, names list)."""
    n = ctypes.c_int64()
    _check(lib().fnn_phylip_taxa(str(path).encode(), ctypes.byref(n)))
    n = n.value
    D = np.empty((n, n), dtype=np.float64)
    names = ctypes.create_string_buffer(n * name_len)
    _check(lib().fnn_read_phylip(str(path).encode(), n, _dp(D), names, name_len, int(threads)))
    raw = names.raw
    return D, [raw[i * name_len:(i + 1) * name_len].split(b"\0", 1)[0].decode("ascii", "replace") for i in range(n)]


def read_alignment(path, threads=0, name_len=64):
    """Native FASTA / sequential PHYLIP alignment loader (fnn_alignment_size + fnn_read_alignment; host only, no device
    needed).  Returns (codes[n, L] uint8 with A=0 C=1 G=2 T=3 and 4 = missing, names list)."""
    n, L = ctypes.c_int64(), ctypes.c_int64()
    _check(lib().fnn_alignment_size(str(path).encode(), ctypes.byref(n), ctypes.byref(L)))
    n, L = n.value, L.value
    codes = np.empty((n, L), dtype=np.uint8)
    names = ctypes.create_string_buffer(n * name_len)
    _check(lib().fnn_read_alignment(str(path).encode(), n, L, codes.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), names, name_len,
                                    int(threads)))
    raw = names.raw
    return codes, [raw[i * name_len:(i + 1) * name_len].split(b"\0", 1)[0].decode("ascii", "replace") for i in range(n)]


def distances(codes, model="p", undefined=None, **opts):
    """fnn_distances: the [n, n] float64 distance matrix of an [n, L] code array, computed on the device.
    model: "p" | "jc69" | "k2p"; undefined=None: an undefined pair (no comparable site, saturation) is an error naming the
    first such pair; a finite value >= 0 is stored there instead."""
    codes, m, u = _alignment_args(codes, model, undefined)
    o = default_opts(**opts)
    n, L = codes.shape
    D = np.empty((n, n), dtype=np.float64)
    _check(lib().fnn_distances(ctypes.byref(o), codes.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), n, L, m, u, _dp(D)))
    return D


def java_double_str(v):
    """Double.toString(v) as the Nexus writer prints it."""
    buf = ctypes.create_string_buffer(40)
    _check(lib().fnn_java_double_to_string(float(v), buf, 40))
    return buf.value.decode()


def write_nexus(path, ordering, split_i, split_j, weight, D=None, names=None, threads=0):
    """fnn_write_nexus: the output of OutputPrinter.NexusWithSplitsAndDistances for the kept splits (host only)."""
    ordering = np.ascontiguousarray(ordering, dtype=np.int32)
    n = ordering.shape[0] - 1
    si = np.ascontiguousarray(split_i, dtype=np.int32)
    sj = np.ascontiguousarray(split_j, dtype=np.int32)
    w = np.ascontiguousarray(weight, dtype=np.float64)
    ip = ctypes.POINTER(ctypes.c_int32)
    nbuf, stride = None, 0
    if names is not None:
        enc = [str(s).encode("ascii", "replace") for s in names]
        stride = max(len(e) for e in enc) + 1
        nbuf = b"".join(e.ljust(stride, b"\0") for e in enc)
    Dp = None
    if D is not None:
        D = np.ascontiguousarray(D, dtype=np.float64)
        Dp = _dp(D)
    _check(lib().fnn_write_nexus(None if path is None else str(path).encode(), n, nbuf, stride, Dp, ordering.ctypes.data_as(ip),
                                 si.ctypes.data_as(ip), sj.ctypes.data_as(ip), _dp(w), len(w), int(threads)))


def network(D, cutoff=1e-6, **opts):
    """fnn_network: ordering + split weights + split emission in one call, distances kept on the device.
    Returns (ordering, split_i, split_j, weight)."""
    D = np.ascontiguousarray(D, dtype=np.float64)
    n = D.shape[0]
    o = default_opts(**opts)
    cap = n * (n - 1) // 2
    ordering = np.zeros(n + 1, dtype=np.int32)
    si, sj, w = np.zeros(cap, dtype=np.int32), np.zeros(cap, dtype=np.int32), np.zeros(cap, dtype=np.float64)
    kept = ctypes.c_int64()
    ip = ctypes.POINTER(ctypes.c_int32)
    _check(lib().fnn_network(ctypes.byref(o), _dp(D), n, float(cutoff), ordering.ctypes.data_as(ip), si.ctypes.data_as(ip),
                             sj.ctypes.data_as(ip), _dp(w), cap, ctypes.byref(kept)))
    k = kept.value
    return ordering, si[:k].copy(), sj[:k].copy(), w[:k].copy()


def csw_matvec(which, v, n, variant="default", **opts):
    """which: 'ab' | 'atx' | 'unconstrained' on a packed npairs vector (fnn_csw_matvec)."""
    opts = dict(opts, csw_variant=CSW_VARIANTS[variant])
    v = np.ascontiguousarray(v, dtype=np.float64)
    o = default_opts(**opts)
    out = np.zeros_like(v)
    _check(lib().fnn_csw_matvec(ctypes.byref(o), {"ab": 0, "atx": 1, "unconstrained": 2}[which], _dp(v), int(n), _dp(out)))
    return out


def weighted_splits(ordering, x, cutoff=1e-6):
    """Split emission of FastNN.java:455-466: keep x > cutoff in (i,j) row-major-upper order; split (i,j) is the taxon
    set {ordering[i+1..j]}.  Returns a list of (sorted taxon list, weight); sets are built only for kept splits."""
    n = len(ordering) - 1
    out = []
    idx = 0
    for i in range(n):
        row = x[idx: idx + (n - 1 - i)]
        for off in np.nonzero(row > cutoff)[0]:
            j = i + 1 + int(off)
            out.append((sorted(int(t) for t in ordering[i + 1: j + 1]), float(row[off])))
        idx += n - 1 - i
    return out


class _NetMaker:
    """Shape of NetMakerOriginal (NetMakerOriginal.java:51,129): construct with D, call runNeighborNet()."""

    _mode = "canonical"

    def __init__(self, D, numTaxa, numThreads=1, pool=None, **opts):
        self.D = D
        self.ntax = int(numTaxa)
        self.opts = dict(opts)
        self.opts.setdefault("mode", self._mode)
        self.ordering = None

    def runNeighborNet(self):
        self.ordering = order(np.asarray(self.D, dtype=np.float64)[: self.ntax, : self.ntax], **self.opts)
        return self.ordering

    def getOrdering(self):
        return self.ordering


class NeighborNetCanonical(_NetMaker):
    """NeighborNetCanonical.java:34."""


class NeighborNetLocal(_NetMaker):
    """NeighborNetLocal.java:26 (relaxed); `additive` as in the reference constructor."""

    def __init__(self, D, numTaxa, numThreads=1, additive=False, pool=None, **opts):
        super().__init__(D, numTaxa, numThreads, pool, mode="relaxed", additive=int(bool(additive)), **opts)


class NeighborNetRandom(_NetMaker):
    """NeighborNetRandom.java:24; myAmount in {"LOGN","N","NLOGN"}, multiplier as -mult."""

    def __init__(self, D, numTaxa, numThreads=1, pool=None, myAmount="NLOGN", multiplier=5, **opts):
        super().__init__(D, numTaxa, numThreads, pool, mode="random_" + myAmount.lower(), mult=int(multiplier), **opts)
