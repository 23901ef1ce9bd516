"""ctypes bindings for the interval-censored MHRS restatement, oracle/pht_oracle_iv.c (TEST INFRASTRUCTURE ONLY, under
the same rule as pyoracle.py: nothing under phasetype_b200/ imports it).

The library is built next to libphtoracle.so, with the same compiler flags as oracle/Makefile, into
oracle/_build/libphtoracle_iv.so: by build() (called from __graft_entry__.build()), or on first use when it is missing.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import scipy

from oracle import pyoracle as po

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "pht_oracle_iv.c")
SO = os.path.join(HERE, "_build", "libphtoracle_iv.so")
# the flags of oracle/Makefile: no compiler-made FMAs, so host rounding equals the device's (-fmad=false)
CFLAGS = ["-O2", "-std=gnu11", "-fPIC", "-ffp-contract=off", "-mfma", "-fno-math-errno", "-Wall", "-Wno-unused-variable",
          "-Wno-unused-but-set-variable", "-Wno-unused-function"]
DEPS = [SRC, os.path.join(HERE, "pht_oracle.c"), os.path.join(HERE, "pht_oracle.h"),
        os.path.join(HERE, "..", "phasetype_b200", "csrc", "pht_math.h"), os.path.join(HERE, "..", "phasetype_b200", "csrc", "pht_philox.h"),
        os.path.join(HERE, "..", "phasetype_b200", "csrc", "pht_eigen.h")]

_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_lp = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
_up = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")


def build():
    """gcc, linked like libphtoracle.so against scipy's OpenBLAS (the restatement's LAPACK calls); skipped when up to date."""
    if os.path.exists(SO) and all(os.path.getmtime(d) <= os.path.getmtime(SO) for d in DEPS if os.path.exists(d)):
        return SO
    obdir = os.path.join(os.path.dirname(os.path.dirname(scipy.__file__)), "scipy.libs")
    oblib = next(f for f in sorted(os.listdir(obdir)) if f.startswith("libscipy_openblas") and f.endswith(".so"))
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    subprocess.run(["gcc"] + CFLAGS + ["-shared", "-Wl,-Bsymbolic", "-o", SO, SRC, "-L" + obdir, "-l:" + oblib,
                                        "-Wl,-rpath," + obdir, "-lm"], check=True)
    return SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(SO)
        L.pho_mhrs_paths_iv.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_long, C.c_long, _dp, _ip, _dp, C.c_int,
                                        _dp, _dp, _dp, C.c_int, _ip, _ip, _dp, _up]
        L.pho_sweep_stats_iv.argtypes = [C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int, _ip, _dp,
                                         _dp, _dp, C.c_long, _ip, _dp, C.c_int, C.c_int, C.c_int, _lp, _lp, _lp, _up]
        _lib = L
    return _lib


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def mhrs_paths_iv(seed, it, y, cens, u, S, s, mhit=1, obs0=0, stride=1):
    """po.mhrs_paths("oracle", ...) for interval-censored data: observation k's absorption time lies in [y[k], u[k]]
    (u = +inf: no bound).  Returns (B, N, z, counters)."""
    y = _f64(y); cens = _i32(cens); u = _f64(u); S = _f64(S); s = _f64(s)
    n = s.shape[0]; count = y.shape[0]
    _, Pfull = po.embedded(S, s)
    cnt = np.zeros(po.N_COUNTERS, dtype=np.uint64)
    B = np.zeros(count, dtype=np.int32); N = np.zeros(count * n * n, dtype=np.int32); z = np.zeros(count * n)
    rc = lib().pho_mhrs_paths_iv(seed, it, obs0, stride, count, y, cens, u, n, S, s, Pfull, mhit, B, N, z, cnt)
    if rc != 0:
        raise RuntimeError("pho_mhrs_paths_iv failed rc=%d" % rc)
    return B, N.reshape(count, n * n), z.reshape(count, n), po._counters(cnt)


def sweep_stats_iv(seed, it, first, mhit, n, T, Cm, theta, y, cens, u, zbits, rank=0, world=1):
    """po.sweep_stats(...) of method MHRS for interval-censored data (u as in mhrs_paths_iv)."""
    y = _f64(y); cens = _i32(cens); u = _f64(u); theta = _f64(theta)
    T = _i32(np.asarray(T).ravel()); Cm = _f64(np.asarray(Cm).ravel())
    N = np.zeros(n * n, dtype=np.int64); B = np.zeros(n, dtype=np.int64); z = np.zeros(n, dtype=np.int64)
    cnt = np.zeros(po.N_COUNTERS, dtype=np.uint64)
    rc = lib().pho_sweep_stats_iv(seed, it, 1 if first else 0, mhit, n, theta.shape[0], T, Cm, theta, y, y.shape[0], cens, u,
                                  rank, world, zbits, N, B, z, cnt)
    if rc != 0:
        raise RuntimeError("pho_sweep_stats_iv failed rc=%d" % rc)
    return N, B, z, po._counters(cnt)


def gibbs_iv(seed, it, mhit, n, nu, zeta, T, Cm, y, cens, u, start, zbits):
    """The MHRS chain for interval-censored data from the CPU restatement: sweep_stats_iv + po.update per sweep,
    (it, m) array like LJMA_Gibbs's res with row 0 = start."""
    theta = _f64(start).copy(); m = theta.shape[0]
    res = np.zeros((it, m)); res[0] = theta
    for i in range(1, it):
        N, _, z, _ = sweep_stats_iv(seed, i, i == 1, mhit, n, T, Cm, theta, y, cens, u, zbits)
        theta = po.update(seed, i, n, nu, zeta, T, Cm, zbits, N, z)
        res[i] = theta
    return res
