"""ctypes bindings for the delayed-entry restatement, oracle/pht_oracle_entry.c (TEST INFRASTRUCTURE ONLY, under the same
rule as pyoracle.py: nothing under phasetype_b200/ imports it).

The library is built next to libphtoracle.so, with the same compiler flags as oracle/Makefile, into
oracle/_build/libphtoracle_entry.so: by build() (called from __graft_entry__.build()), or on first use when it is missing.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import scipy

from oracle import pyoracle as po
from oracle import pyoracle_iv as poi
from oracle import pyoracle_unif as pu

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "pht_oracle_entry.c")
SO = os.path.join(HERE, "_build", "libphtoracle_entry.so")
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
        L.pho_log1p.restype = C.c_double; L.pho_log1p.argtypes = [C.c_double]
        L.pho_log1p_general.restype = C.c_double; L.pho_log1p_general.argtypes = [C.c_double]
        L.pho_entry_tables.argtypes = [C.c_int, _dp, _dp, _dp, C.c_double, C.c_int, _dp]
        L.pho_entry_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_long, C.c_long, _dp, _ip, C.c_void_p, _dp,
                                      C.c_void_p, C.c_int, _dp, _dp, C.c_int, _ip, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p]
        L.pho_entry_sweep_stats.argtypes = [C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int, _ip, _dp, _dp, _dp, C.c_long,
                                            _ip, C.c_void_p, _dp, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, _lp, _lp, _lp]
        _lib = L
    return _lib


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return None if a is None else a.ctypes.data


def log1p(x):
    return lib().pho_log1p(float(x))


def log1p_general(x):
    return lib().pho_log1p_general(float(x))


def entry_tables(S, s, pi=None, tmax=1.0, cap=CAP):
    """(sigma, phi) for k <= K_sweep of the table at tmax: S(a) = sum_k Pois(k; lam a) sigma_k, F(a) likewise with phi."""
    S = _f64(S); s = _f64(s); n = s.shape[0]
    pi = _f64(pi) if pi is not None else np.eye(n)[0]
    etab = np.zeros(2 * cap)
    K = lib().pho_entry_tables(n, S, s, pi, float(tmax), cap, etab)
    if K < 0:
        raise RuntimeError("pho_entry_tables: tmax beyond the table")
    return etab[:K + 1].copy(), etab[cap:cap + K + 1].copy()


def entry_paths(seed, it, y, cens, a, S, s, u=None, pi=None, obs0=0, stride=1, paths=True, cap=CAP):
    """Ghost counts M of the observations (entry ages a), and with paths their ghost paths in (observation, ghost index)
    order.  Returns (M, B, N, z, err) with err the engine's error bits (0 when all went well)."""
    y = _f64(y); cens = np.ascontiguousarray(cens, dtype=np.int32); a = _f64(a); S = _f64(S); s = _f64(s)
    u = None if u is None else _f64(u); pi = None if pi is None else _f64(pi)
    n = s.shape[0]; count = y.shape[0]
    M = np.zeros(max(count, 1), dtype=np.int32)
    err = lib().pho_entry_paths(seed, it, obs0, stride, count, y, cens, _ptr(u), a, _ptr(pi), n, S, s, cap, M, 0, None, None, None)
    M = M[:count]
    if not paths or err:
        return M, None, None, None, int(err)
    G = int(M.astype(np.int64).sum())
    B = np.zeros(max(G, 1), dtype=np.int32); N = np.zeros(max(G, 1) * n * n, dtype=np.int32); z = np.zeros(max(G, 1) * n)
    M2 = np.zeros(max(count, 1), dtype=np.int32)
    err = lib().pho_entry_paths(seed, it, obs0, stride, count, y, cens, _ptr(u), a, _ptr(pi), n, S, s, cap, M2, G,
                                B.ctypes.data, N.ctypes.data, z.ctypes.data)
    return M, B[:G], N[:G * n * n].reshape(G, n * n), z[:G * n].reshape(G, n), int(err)


def entry_sweep_stats(seed, it, first, n, T, Cm, theta, y, cens, a, zbits, u=None, pi=None, rank=0, world=1, cap=CAP):
    """One sweep's (N, B, zfix) of the shard {k : k % world == rank} with the ghosts of its truncated observations, as
    pht_engine_sweep_stats returns them."""
    y = _f64(y); cens = np.ascontiguousarray(cens, dtype=np.int32); a = _f64(a); theta = _f64(theta)
    u = None if u is None else _f64(u); pi = None if pi is None else _f64(pi)
    T = np.ascontiguousarray(np.asarray(T).ravel(), dtype=np.int32); Cm = _f64(np.asarray(Cm).ravel())
    N = np.zeros(n * n, dtype=np.int64); B = np.zeros(n, dtype=np.int64); z = np.zeros(n, dtype=np.int64)
    err = lib().pho_entry_sweep_stats(seed, it, 1 if first else 0, n, theta.shape[0], T, Cm, theta, y, y.shape[0], cens,
                                      _ptr(u), a, _ptr(pi), rank, world, zbits, cap, N, B, z)
    if err:
        raise RuntimeError("pho_entry_sweep_stats: error bits %d" % err)
    return N, B, z


def gibbs_entry(seed, it, n, nu, zeta, T, Cm, y, cens, a, start, zbits, u=None):
    """The method-64 chain with entry ages from the host restatement: entry_sweep_stats + po.update per sweep, (it, m)
    array like LJMA_Gibbs's res with row 0 = start (pi = e1)."""
    theta = _f64(start).copy(); m = theta.shape[0]
    res = np.zeros((it, m)); res[0] = theta
    for i in range(1, it):
        N, _, z = entry_sweep_stats(seed, i, i == 1, n, T, Cm, theta, y, cens, a, zbits, u=u)
        theta = po.update(seed, i, n, nu, zeta, T, Cm, zbits, N, z)
        res[i] = theta
    return res
