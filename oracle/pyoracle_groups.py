"""ctypes bindings for the groups restatement, oracle/pht_oracle_groups.c (TEST INFRASTRUCTURE ONLY, under the same rule as
pyoracle.py: nothing under phasetype_b200/ imports it).

The library is built next to libphtoracle.so, with the same compiler flags as oracle/Makefile, into
oracle/_build/libphtoracle_groups.so: by build() (called from __graft_entry__.build()), or on first use when it is missing.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import scipy

from oracle import pyoracle_iv as poi
from oracle import pyoracle_unif as pu

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "pht_oracle_groups.c")
SO = os.path.join(HERE, "_build", "libphtoracle_groups.so")
DEPS = pu.DEPS + [SRC, os.path.join(HERE, "pht_oracle_unif.c")]
CAP = pu.CAP

_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_lp = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")


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
        L.pho_groups_sweep_stats.argtypes = [C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int, _ip, _dp, _dp, _dp, C.c_long,
                                             _ip, C.c_void_p, _ip, C.c_void_p, C.c_int, C.c_int, _lp, _lp, _lp]
        L.pho_groups_update.argtypes = [C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int, _dp, _dp, _ip, _dp, C.c_int,
                                        _lp, _lp, _dp]
        _lib = L
    return _lib


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return None if a is None else a.ctypes.data


def _structs(T, Cm, n):
    T = np.ascontiguousarray(np.asarray(T, dtype=np.int32).reshape(-1, (n + 1) ** 2))
    Cm = np.ascontiguousarray(np.asarray(Cm, dtype=np.float64).reshape(-1, (n + 1) ** 2))
    return T, Cm


def groups_sweep_stats(seed, it, first, n, T, Cm, theta, y, cens, group, zbits, u=None, pi=None, cap=CAP):
    """One sweep's per-group (N (G, n*n), B (G, n), zfix (G, n)) of a single-rank data set, as pht_engine_group_stats
    returns them.  T, Cm: (G, (n+1)^2) column-major structures; group[k] in 0..G-1."""
    T, Cm = _structs(T, Cm, n)
    G = T.shape[0]
    y = _f64(y); cens = np.ascontiguousarray(cens, dtype=np.int32); theta = _f64(theta)
    group = np.ascontiguousarray(group, dtype=np.int32)
    u = None if u is None else _f64(u); pi = None if pi is None else _f64(pi)
    N = np.zeros(G * n * n, dtype=np.int64); B = np.zeros(G * n, dtype=np.int64); z = np.zeros(G * n, dtype=np.int64)
    err = lib().pho_groups_sweep_stats(seed, it, 1 if first else 0, n, G, T.ravel(), Cm.ravel(), theta, y, y.shape[0], cens,
                                       _ptr(u), group, _ptr(pi), zbits, cap, N, B, z)
    if err:
        raise RuntimeError("pho_groups_sweep_stats: error bits %d" % err)
    return N.reshape(G, n * n), B.reshape(G, n), z.reshape(G, n)


def groups_update(seed, it, n, nu, zeta, T, Cm, zbits, N, zfix):
    """The grouped gather (groups ascending, cells in the reference's order within each) and the Gamma draw of theta."""
    T, Cm = _structs(T, Cm, n)
    nu = _f64(nu); zeta = _f64(zeta)
    out = np.zeros(nu.shape[0])
    lib().pho_groups_update(seed, it, n, nu.shape[0], T.shape[0], nu, zeta, T.ravel(), Cm.ravel(), zbits,
                            np.ascontiguousarray(N, dtype=np.int64).ravel(), np.ascontiguousarray(zfix, dtype=np.int64).ravel(), out)
    return out


def gibbs_groups(seed, it, n, nu, zeta, T, Cm, y, cens, group, start, zbits, u=None):
    """The grouped method-64 chain from the host restatement: groups_sweep_stats + groups_update per sweep, (it, m) array
    like LJMA_Gibbs's res with row 0 = start (pi = e1)."""
    theta = _f64(start).copy(); m = theta.shape[0]
    res = np.zeros((it, m)); res[0] = theta
    for i in range(1, it):
        N, _, z = groups_sweep_stats(seed, i, i == 1, n, T, Cm, theta, y, cens, group, zbits, u=u)
        theta = groups_update(seed, i, n, nu, zeta, T, Cm, zbits, N, z)
        res[i] = theta
    return res
