"""oracle.dist — CPU restatement of the alignment distances (dist_oracle.cpp).  TEST INFRASTRUCTURE ONLY.

Its own small library, libdist_oracle.so, built with the flags of the ordering oracle (-ffp-contract=off: no FMA
contraction, so csrc/fnn_log.h gives the bits the device gives).  build() writes it next to this file; where that
directory is read-only, lib() builds a private copy in the temporary directory instead.
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRCS = [os.path.join(_HERE, "dist_oracle.cpp"),
         os.path.join(os.path.dirname(_HERE), "fastneighbornet_b200", "csrc", "fnn_log.h")]
_LIB = None

MODELS = {"p": 0, "jc69": 1, "k2p": 2}


def _compile(out):
    cmd = [os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-pthread",
           "-Wall", "-Wextra", "-shared", "-o", out, _SRCS[0]]
    subprocess.check_call(cmd)


def _stale(so):
    return not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in _SRCS)


def build():
    """Compile libdist_oracle.so next to this file (when missing or older than its sources)."""
    so = os.path.join(_HERE, "libdist_oracle.so")
    if _stale(so):
        _compile(so)
    return so


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(_HERE, "libdist_oracle.so")
        if _stale(so):
            if os.access(_HERE, os.W_OK):
                build()
            else:
                digest = hashlib.sha256(b"".join(open(s, "rb").read() for s in _SRCS)).hexdigest()[:16]
                so = os.path.join(tempfile.gettempdir(), f"fnn_dist_oracle_{os.getuid()}_{digest}.so")
                if not os.path.exists(so):
                    tmp = f"{so}.{os.getpid()}.tmp"
                    _compile(tmp)
                    os.replace(tmp, so)
        L = ctypes.CDLL(so)
        c_dp, c_lp = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64)
        L.oracle_fnn_log.argtypes = [c_dp, ctypes.c_int64, c_dp]
        L.oracle_fnn_log.restype = None
        L.oracle_distances.argtypes = [ctypes.POINTER(ctypes.c_uint8), ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_double,
                                       c_lp, ctypes.c_int64, c_dp, c_lp]
        L.oracle_distances.restype = ctypes.c_int
        _LIB = L
    return _LIB


def _dp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def _lp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))


def fnn_log(x):
    """csrc/fnn_log.h compiled for the host: the logarithm of the alignment distances, elementwise on a float64 array."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty_like(x)
    lib().oracle_fnn_log(_dp(x), x.size, _dp(out))
    return out


def distances(codes, model="p", undefined=None, rows=None):
    """CPU restatement of fnn_distances on the listed rows (default: all).
    Returns (D_rows[len(rows), n] float64, first) with first = (i, j, v, m, s) of the first undefined pair among those rows
    or None; with undefined=None undefined entries hold NaN."""
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    n, L = codes.shape
    rows = np.arange(n, dtype=np.int64) if rows is None else np.ascontiguousarray(rows, dtype=np.int64)
    out = np.empty((rows.shape[0], n), dtype=np.float64)
    first = np.zeros(5, dtype=np.int64)
    rc = lib().oracle_distances(codes.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), n, L, MODELS[model],
                                float("nan") if undefined is None else float(undefined), _lp(rows), rows.shape[0], _dp(out),
                                _lp(first))
    if rc != 0:
        raise ValueError("oracle_distances: bad argument (a code > 4 or a row out of range)")
    return out, (None if first[0] < 0 else tuple(int(v) for v in first))
