"""ctypes bindings for the uniformisation sampler's host restatement, oracle/pht_oracle_unif.c (TEST INFRASTRUCTURE ONLY,
under the same rule as pyoracle.py: nothing under phasetype_b200/ imports it).

The library is built next to libphtoracle.so, with the same compiler flags as oracle/Makefile, into
oracle/_build/libphtoracle_unif.so: by build() (called from __graft_entry__.build()), or on first use when it is missing.
"""
import ctypes as C
import os

import numpy as np

from oracle import pyoracle as po
from oracle import pyoracle_iv as poi

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "pht_oracle_unif.c")
SO = os.path.join(HERE, "_build", "libphtoracle_unif.so")
DEPS = poi.DEPS[1:] + [SRC, os.path.join(HERE, "..", "phasetype_b200", "csrc", "pht_unif.h")]
CAP = 4096                     # PHT_UNIF_CAP

_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_lp = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")


def build():
    """gcc with the flags of oracle/Makefile (the restatement's LAPACK calls linked as in pyoracle_iv); skipped when up to date."""
    if os.path.exists(SO) and all(os.path.getmtime(d) <= os.path.getmtime(SO) for d in DEPS if os.path.exists(d)):
        return SO
    import subprocess
    import scipy
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
        L.pho_unif_table.argtypes = [C.c_int, _dp, _dp, _dp, C.c_double, C.c_int, _dp]
        L.pho_unif_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_long, C.c_long, _dp, _ip, C.c_void_p, C.c_void_p,
                                     C.c_int, _dp, _dp, C.c_int, _ip, _ip, _dp]
        L.pho_unif_sweep_stats.argtypes = [C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int, _ip, _dp, _dp, _dp, C.c_long,
                                           _ip, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, _lp, _lp, _lp]
        _lib = L
    return _lib


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return None if a is None else a.ctypes.data


def layout(n, cap=CAP):
    """Offsets (in doubles) of the table pieces, as pht_unif_layout_make."""
    o = 8; L = {}
    for name, size in (("lgk", cap), ("R", n * n), ("r", n), ("P", cap * n * n), ("q", cap * n), ("g", cap * n)):
        L[name] = o; o += size
    L["total"] = o
    return L


def table(S, s, pi=None, tmax=1.0, cap=CAP):
    """The sweep's table for the column-major S (flat) and s.  Returns (K_sweep or -1, dict of lam, lgk, R, r, P, q, g)
    with P as (K+1, n, n) row-major arrays of R^k, q as (K+1, n), g as (K+1, n)."""
    S = _f64(S); s = _f64(s); n = s.shape[0]
    pi = _f64(pi) if pi is not None else np.eye(n)[0]
    L = layout(n, cap)
    tab = np.zeros(L["total"])
    K = lib().pho_unif_table(n, S, s, pi, float(tmax), cap, tab)
    Kt = int(tab[1])
    out = {"lam": tab[0], "lgk": tab[L["lgk"]:L["lgk"] + cap].copy(),
           "R": tab[L["R"]:L["R"] + n * n].reshape(n, n, order="F"), "r": tab[L["r"]:L["r"] + n].copy(),
           "P": tab[L["P"]:L["P"] + (Kt + 1) * n * n].reshape(Kt + 1, n, n).transpose(0, 2, 1),
           "q": tab[L["q"]:L["q"] + (Kt + 1) * n].reshape(Kt + 1, n), "g": tab[L["g"]:L["g"] + (Kt + 1) * n].reshape(Kt + 1, n)}
    return K, out


def truncation(x):
    """K(x) = ceil(x + 10 sqrt(x) + 20), the last power a sum at Poisson mean x uses."""
    v = x + 10.0 * np.sqrt(x) + 20.0
    return int(np.ceil(v))


def unif_paths(seed, it, y, cens, S, s, u=None, pi=None, obs0=0, stride=1, cap=CAP):
    """Per-observation paths of the uniformisation sampler (u: upper bounds, +inf = none; pi: start distribution,
    default e1).  Returns (B, N, z, err) with err the engine's error bits (0 when all went well)."""
    y = _f64(y); cens = np.ascontiguousarray(cens, dtype=np.int32); S = _f64(S); s = _f64(s)
    u = None if u is None else _f64(u); pi = None if pi is None else _f64(pi)
    n = s.shape[0]; count = y.shape[0]
    B = np.zeros(count, dtype=np.int32); N = np.zeros(count * n * n, dtype=np.int32); z = np.zeros(count * n)
    err = lib().pho_unif_paths(seed, it, obs0, stride, count, y, cens, _ptr(u), _ptr(pi), n, S, s, cap, B, N, z)
    return B, N.reshape(count, n * n), z.reshape(count, n), int(err)


def unif_sweep_stats(seed, it, first, n, T, Cm, theta, y, cens, zbits, u=None, pi=None, rank=0, world=1, cap=CAP):
    """One sweep's (N, B, zfix) of the shard {k : k % world == rank}, as pht_engine_sweep_stats returns them."""
    y = _f64(y); cens = np.ascontiguousarray(cens, dtype=np.int32); theta = _f64(theta)
    u = None if u is None else _f64(u); pi = None if pi is None else _f64(pi)
    T = np.ascontiguousarray(np.asarray(T).ravel(), dtype=np.int32); Cm = _f64(np.asarray(Cm).ravel())
    N = np.zeros(n * n, dtype=np.int64); B = np.zeros(n, dtype=np.int64); z = np.zeros(n, dtype=np.int64)
    err = lib().pho_unif_sweep_stats(seed, it, 1 if first else 0, n, theta.shape[0], T, Cm, theta, y, y.shape[0], cens,
                                     _ptr(u), _ptr(pi), rank, world, zbits, cap, N, B, z)
    if err:
        raise RuntimeError("pho_unif_sweep_stats: error bits %d" % err)
    return N, B, z


def gibbs_unif(seed, it, n, nu, zeta, T, Cm, y, cens, start, zbits, u=None):
    """The method-64 chain from the host restatement: unif_sweep_stats + po.update per sweep, (it, m) array like
    LJMA_Gibbs's res with row 0 = start (pi = e1)."""
    theta = _f64(start).copy(); m = theta.shape[0]
    res = np.zeros((it, m)); res[0] = theta
    for i in range(1, it):
        N, _, z = unif_sweep_stats(seed, i, i == 1, n, T, Cm, theta, y, cens, zbits, u=u)
        theta = po.update(seed, i, n, nu, zeta, T, Cm, zbits, N, z)
        res[i] = theta
    return res
