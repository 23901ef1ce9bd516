"""ctypes binding of the panel form of the uniformisation sampler, oracle/pht_oracle_panel.c (TEST INFRASTRUCTURE ONLY, under
the same rule as pyoracle.py: nothing under phasetype_b200/ imports it).

The library is built next to libphtoracle_unif.so, with the same compiler flags, into oracle/_build/libphtoracle_panel.so:
by build() (called from __graft_entry__.build()), or on first use when it is missing.
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
SRC = os.path.join(HERE, "pht_oracle_panel.c")
SO = os.path.join(HERE, "_build", "libphtoracle_panel.so")
DEPS = pu.DEPS + [SRC, os.path.join(HERE, "pht_oracle_unif.c")]
CAP = pu.CAP

_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_ip = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_lp = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
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
        L.pho_panel_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_void_p, _dp, _ip, C.c_void_p, C.c_void_p, _lp, _dp,
                                      _u32p, C.c_int, _dp, _dp, C.c_int, C.c_double, _ip, _ip, _dp, C.c_void_p]
        L.pho_panel_sweep_stats.argtypes = [C.c_uint64, C.c_uint32, C.c_int, C.c_int, _ip, _dp, _dp, C.c_long, _dp, _ip,
                                            C.c_void_p, C.c_void_p, _lp, _dp, _u32p, C.c_int, C.c_int, _lp, _lp, _lp]
        _lib = L
    return _lib


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return None if a is None else a.ctypes.data


def _visits(offsets, t, mask):
    off = np.ascontiguousarray(offsets, dtype=np.int64)
    vt = _f64(t) if len(t) else np.zeros(1)
    vm = np.ascontiguousarray(mask, dtype=np.uint32) if len(mask) else np.zeros(1, dtype=np.uint32)
    return off, vt, vm


def panel_paths(seed, it, y, cens, offsets, t, mask, S, s, u=None, pi=None, obs=None, tmax=0.0, states=False, cap=CAP):
    """Paths of observations with visits (t, mask)[offsets[k]:offsets[k + 1]] (none: the plain sampler), observation k on
    the stream of global observation obs[k] (default k); the table spans tmax (<= 0: the observations).  Returns
    (B, N, z, err), and with states=True (B, N, z, X, err), X the drawn visit states laid out like t."""
    y = _f64(y); cens = np.ascontiguousarray(cens, dtype=np.int32); S = _f64(S); s = _f64(s)
    u = None if u is None else _f64(u); pi = None if pi is None else _f64(pi)
    obs = None if obs is None else np.ascontiguousarray(obs, dtype=np.uint32)
    off, vt, vm = _visits(offsets, t, mask)
    n = s.shape[0]; count = y.shape[0]
    B = np.zeros(max(count, 1), dtype=np.int32); N = np.zeros(max(count, 1) * n * n, dtype=np.int32); z = np.zeros(max(count, 1) * n)
    X = np.zeros(max(int(off[-1]), 1), dtype=np.int32)
    err = lib().pho_panel_paths(seed, it, count, _ptr(obs), y, cens, _ptr(u), _ptr(pi), off, vt, vm, n, S, s, cap, float(tmax),
                                B, N, z, X.ctypes.data)
    out = (B[:count], N[:count * n * n].reshape(count, n * n), z[:count * n].reshape(count, n))
    return out + ((X[:int(off[-1])], int(err)) if states else (int(err),))


def panel_sweep_stats(seed, it, first, n, T, Cm, theta, y, cens, offsets, t, mask, zbits, u=None, pi=None, cap=CAP):
    """One sweep's (N, B, zfix) of a single-rank data set with visits, as pht_engine_sweep_stats returns them."""
    y = _f64(y); cens = np.ascontiguousarray(cens, dtype=np.int32); theta = _f64(theta)
    u = None if u is None else _f64(u); pi = None if pi is None else _f64(pi)
    T = np.ascontiguousarray(np.asarray(T).ravel(), dtype=np.int32); Cm = _f64(np.asarray(Cm).ravel())
    off, vt, vm = _visits(offsets, t, mask)
    N = np.zeros(n * n, dtype=np.int64); B = np.zeros(n, dtype=np.int64); z = np.zeros(n, dtype=np.int64)
    err = lib().pho_panel_sweep_stats(seed, it, 1 if first else 0, n, T, Cm, theta, y.shape[0], y, cens, _ptr(u), _ptr(pi),
                                      off, vt, vm, zbits, cap, N, B, z)
    if err:
        raise RuntimeError("pho_panel_sweep_stats: error bits %d" % err)
    return N, B, z


def gibbs_panel(seed, it, n, nu, zeta, T, Cm, y, cens, offsets, t, mask, start, zbits, u=None, pi=None, beta=None):
    """The method-64 chain with visits from the host restatement: panel_sweep_stats + po.update per sweep, and with beta
    the Dirichlet update of pi (n Gamma(beta_i + B_i, 1) draws on parameter sub-streams m + i, normalised in index order,
    as k_update).  Returns (theta rows (it, m) with row 0 = start, pi rows (it, n) with row 0 = the start pi)."""
    theta = _f64(start).copy(); m = theta.shape[0]
    pi = np.eye(n)[0] if pi is None else _f64(pi).copy()
    res = np.zeros((it, m)); res[0] = theta
    pis = np.zeros((it, n)); pis[0] = pi
    for i in range(1, it):
        N, B, z = panel_sweep_stats(seed, i, i == 1, n, T, Cm, theta, y, cens, offsets, t, mask, zbits, u=u, pi=pi)
        theta = po.update(seed, i, n, nu, zeta, T, Cm, zbits, N, z)
        if beta is not None:
            g = [po.rgamma_at(seed, i, m + k, float(beta[k]) + float(B[k]), 1.0) for k in range(n)]
            tot = 0.0
            for v in g:
                tot += v
            pi = np.array([v / tot for v in g])
        res[i] = theta; pis[i] = pi
    return res, pis
