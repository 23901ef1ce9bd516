"""ctypes binding of the record form of the uniformisation sampler, oracle/pht_oracle_counts.c (TEST INFRASTRUCTURE ONLY,
under the same rule as pyoracle.py: nothing under phasetype_b200/ imports it).

The library is built next to libphtoracle_unif.so, with the same compiler flags, into oracle/_build/libphtoracle_counts.so:
by build() (called from __graft_entry__.build()), or on first use when it is missing.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import scipy

from oracle import pyoracle_iv as poi
from oracle import pyoracle_unif as pu

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "pht_oracle_counts.c")
SO = os.path.join(HERE, "_build", "libphtoracle_counts.so")
DEPS = pu.DEPS + [SRC]
CAP = pu.CAP

_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")


def build():
    """gcc with the flags of oracle/Makefile, linked like pyoracle_unif; skipped when up to date."""
    if os.path.exists(SO) and all(os.path.getmtime(d) <= os.path.getmtime(SO) for d in DEPS if os.path.exists(d)):
        return SO
    obdir = os.path.join(os.path.dirname(os.path.dirname(scipy.__file__)), "scipy.libs")
    oblib = next(f for f in sorted(os.listdir(obdir)) if f.startswith("libscipy_openblas") and f.endswith(".so"))
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    subprocess.run(["gcc"] + poi.CFLAGS + ["-shared", "-Wl,-Bsymbolic", "-o", SO, SRC, "-L" + obdir, "-l:" + oblib,
                                            "-Wl,-rpath," + obdir, "-lm"], check=True)
    return SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(SO)
        L.pho_unif_record_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, _dp, _ip, C.c_void_p, C.c_void_p, _u32p,
                                            C.c_int, _dp, _dp, C.c_int, C.c_int, _ip, _ip, _dp]
        _lib = L
    return _lib


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return None if a is None else a.ctypes.data


def record_paths(seed, it, y, cens, counts, S, s, u=None, pi=None, kb=255, cap=CAP):
    """The record form of the sampler: record k's counts[k] units on the streams of expanded observations base_k + j
    (base: exclusive prefix sum of counts), weights buffered for k <= kb and recomputed beyond.  Returns (B, N, z, err)
    in expanded order, to compare with pyoracle_unif.unif_paths(np.repeat(y, counts), ...)."""
    y = _f64(y); cens = np.ascontiguousarray(cens, dtype=np.int32); S = _f64(S); s = _f64(s)
    counts = np.ascontiguousarray(counts, dtype=np.uint32)
    u = None if u is None else _f64(u); pi = None if pi is None else _f64(pi)
    n = s.shape[0]; total = int(counts.astype(np.int64).sum())
    B = np.zeros(max(total, 1), dtype=np.int32); N = np.zeros(max(total, 1) * n * n, dtype=np.int32); z = np.zeros(max(total, 1) * n)
    err = lib().pho_unif_record_paths(seed, it, y.shape[0], y, cens, _ptr(u), _ptr(pi), counts, n, S, s, cap, int(kb), B, N, z)
    return B[:total], N[:total * n * n].reshape(total, n * n), z[:total * n].reshape(total, n), int(err)
