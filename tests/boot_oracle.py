"""CPU composition of the existing oracles into the bootstrap of fnn_bootstrap (include/fastnn.h, DESIGN.md §4.5).  TEST
INFRASTRUCTURE ONLY.

java_random -> dist.distances (oracle/dist_oracle.cpp) -> order (oracle/nnet_oracle.cpp) -> setup_d + l1_split_weights
(oracle/csw_l1.cpp) -> the splits with x > cutoff.  A split is matched as a bipartition by brute force: both sides of it
normalised to the side without taxon 1, as a sorted tuple, and looked up in a set (not the device's range rule)."""
import concurrent.futures
import os

import numpy as np

import oracle
from oracle import dist as dist_oracle


def packed_to_ij(n, idx):
    """Packed upper-triangle indices (row-major, i < j) -> (i, j) arrays."""
    idx = np.asarray(idx, dtype=np.int64)
    rs = np.array([i * (2 * n - i - 1) // 2 for i in range(n)], dtype=np.int64)
    i = np.searchsorted(rs, idx, side="right") - 1
    return i, idx - rs[i] + i + 1


def split_key(n, members):
    """The side of the bipartition {members, rest} without taxon 1, as a sorted tuple of taxon ids (1-based)."""
    s = set(int(t) for t in members)
    if 1 in s:
        s = set(range(1, n + 1)) - s
    return tuple(sorted(s))


def network(codes, model="p", undefined=None, cutoff=1e-6, mode="canonical", seed=12345, mult=5, fallback=1024):
    """The network of one alignment: dict(ordering, split_i, split_j, weight, cg_iters), or dict(undefined=(i, j, v, m, s))
    when undefined is None and a pair is undefined."""
    D, first = dist_oracle.distances(codes, model, undefined=undefined)
    if undefined is None and first is not None:
        return {"undefined": first}
    n = codes.shape[0]
    o, _, _ = oracle.order(D, mode=mode, seed=seed, mult=mult, fallback=fallback, want_trace=False)
    du = D[np.triu_indices(n, 1)]
    x, st = oracle.l1_split_weights(n, oracle.setup_d(o, du))
    kept = np.nonzero(x > cutoff)[0]
    si, sj = packed_to_ij(n, kept)
    return {"ordering": o, "split_i": si.astype(np.int32), "split_j": sj.astype(np.int32), "weight": x[kept],
            "cg_iters": st["cg_iters"]}


def bootstrap(codes, R, boot_seed, model="p", undefined=None, cutoff=1e-6, mode="canonical", seed=12345, mult=5, fallback=1024):
    """dict(original=network(codes), draws[R, L], replicates=[network of each replicate], support[k]).  With undefined=None
    the list stops at the first replicate with an undefined pair (its entry holds "undefined") and support is None."""
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    n, L = codes.shape
    kw = dict(model=model, undefined=undefined, cutoff=cutoff, mode=mode, seed=seed, mult=mult, fallback=fallback)
    orig = network(codes, **kw)
    draws = oracle.java_random(boot_seed, L, R * L).reshape(R, L)
    out = {"original": orig, "draws": draws, "replicates": [], "support": None}
    if "undefined" in orig:
        return out
    index = {split_key(n, orig["ordering"][i + 1: j + 1]): k for k, (i, j) in enumerate(zip(orig["split_i"], orig["split_j"]))}
    support = np.zeros(len(index), dtype=np.int32)
    # the replicates are independent and ctypes releases the GIL inside the oracles, which keep no shared state here
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(R, os.cpu_count() or 1)) as pool:
        reps = list(pool.map(lambda r: network(codes[:, np.sort(draws[r])], **kw), range(R)))
    for rep in reps:
        out["replicates"].append(rep)
        if "undefined" in rep:
            return out
        for i, j in zip(rep["split_i"], rep["split_j"]):
            k = index.get(split_key(n, rep["ordering"][i + 1: j + 1]))
            if k is not None:
                support[k] += 1
    out["support"] = support
    return out
