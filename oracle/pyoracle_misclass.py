"""ctypes binding of the emission form of the panel sampler, oracle/pht_oracle_misclass.c (TEST INFRASTRUCTURE ONLY, under
the same rule as pyoracle.py: nothing under phasetype_b200/ imports it).

The library is built next to libphtoracle_unif.so, with the same compiler flags, into oracle/_build/libphtoracle_misclass.so:
by build() (called from __graft_entry__.build()), or on first use when it is missing.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import scipy

from oracle import pyoracle as po
from oracle import pyoracle_groups as pg
from oracle import pyoracle_iv as poi
from oracle import pyoracle_unif as pu

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "pht_oracle_misclass.c")
SO = os.path.join(HERE, "_build", "libphtoracle_misclass.so")
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
        L.pho_misclass_paths.argtypes = [C.c_uint64, C.c_uint32, C.c_long, C.c_void_p, _dp, _ip, C.c_void_p, C.c_void_p, _lp,
                                         _dp, _u32p, _dp, C.c_int, C.c_int, _dp, _dp, C.c_int, C.c_double, _ip, _ip, _dp,
                                         C.c_void_p]
        L.pho_misclass_sweep_stats.argtypes = [C.c_uint64, C.c_uint32, C.c_int, C.c_int, _ip, _dp, _dp, C.c_long, C.c_void_p, _dp, _ip,
                                               C.c_void_p, C.c_void_p, _lp, _dp, _u32p, _dp, C.c_int, C.c_int, C.c_int,
                                               _lp, _lp, _lp, _lp]
        _lib = L
    return _lib


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return None if a is None else a.ctypes.data


def _visits(offsets, t, stage):
    off = np.ascontiguousarray(offsets, dtype=np.int64)
    vt = _f64(t) if len(t) else np.zeros(1)
    vs = np.ascontiguousarray(stage, dtype=np.uint32) if len(stage) else np.zeros(1, dtype=np.uint32)
    return off, vt, vs


def misclass_paths(seed, it, y, cens, offsets, t, stage, E, S, s, u=None, pi=None, obs=None, tmax=0.0, states=False, cap=CAP):
    """Paths of observations with stage visits (t, stage)[offsets[k]:offsets[k + 1]] read through E (n, S) (none: the
    plain sampler), S the sub-generator (column-major, as pyoracle_panel.panel_paths takes it).  Returns (B, N, z, err),
    and with states=True (B, N, z, X, err), X the drawn visit states laid out like t."""
    y = _f64(y); cens = np.ascontiguousarray(cens, dtype=np.int32); S = _f64(S); s = _f64(s)
    u = None if u is None else _f64(u); pi = None if pi is None else _f64(pi)
    obs = None if obs is None else np.ascontiguousarray(obs, dtype=np.uint32)
    Em = _f64(E); Sn = int(Em.shape[1])
    off, vt, vs = _visits(offsets, t, stage)
    n = s.shape[0]; count = y.shape[0]
    B = np.zeros(max(count, 1), dtype=np.int32); N = np.zeros(max(count, 1) * n * n, dtype=np.int32); z = np.zeros(max(count, 1) * n)
    X = np.zeros(max(int(off[-1]), 1), dtype=np.int32)
    err = lib().pho_misclass_paths(seed, it, count, _ptr(obs), y, cens, _ptr(u), _ptr(pi), off, vt, vs, Em.ravel(), Sn, n, S, s,
                                   cap, float(tmax), B, N, z, X.ctypes.data)
    out = (B[:count], N[:count * n * n].reshape(count, n * n), z[:count * n].reshape(count, n))
    return out + ((X[:int(off[-1])], int(err)) if states else (int(err),))


def misclass_sweep_stats(seed, it, first, n, T, Cm, theta, y, cens, offsets, t, stage, E, zbits, u=None, pi=None, obs=None,
                         cap=CAP):
    """One sweep's (N, B, zfix, K) of a single-rank data set with stage visits, as pht_engine_sweep_stats and
    pht_engine_emission_stats return them; observation k on the stream of global observation obs[k] (default k)."""
    y = _f64(y); cens = np.ascontiguousarray(cens, dtype=np.int32); theta = _f64(theta)
    u = None if u is None else _f64(u); pi = None if pi is None else _f64(pi)
    T = np.ascontiguousarray(np.asarray(T).ravel(), dtype=np.int32); Cm = _f64(np.asarray(Cm).ravel())
    Em = _f64(E); Sn = int(Em.shape[1])
    off, vt, vs = _visits(offsets, t, stage)
    N = np.zeros(n * n, dtype=np.int64); B = np.zeros(n, dtype=np.int64); z = np.zeros(n, dtype=np.int64)
    K = np.zeros(n * Sn, dtype=np.int64)
    obs = None if obs is None else np.ascontiguousarray(obs, dtype=np.uint32)
    err = lib().pho_misclass_sweep_stats(seed, it, 1 if first else 0, n, T, Cm, theta, y.shape[0], _ptr(obs), y, cens, _ptr(u), _ptr(pi),
                                         off, vt, vs, Em.ravel(), Sn, zbits, cap, N, B, z, K)
    if err:
        raise RuntimeError("pho_misclass_sweep_stats: error bits %d" % err)
    return N, B, z, K.reshape(n, Sn)


def _group_stats(seed, i, n, T, Cm, theta, y, cens, offsets, t, stage, E, zbits, u, pi, group):
    """misclass_sweep_stats per group on the group's own structure (T, Cm: (G, (n+1)^2)), every observation on its own
    stream: (N (G, n*n), B summed, zfix (G, n), K summed)."""
    T, Cm = pg._structs(T, Cm, n)
    off = np.asarray(offsets, dtype=np.int64); t = np.asarray(t); stage = np.asarray(stage)
    Ns, zs, B, K = [], [], 0, 0
    for g in range(T.shape[0]):
        idx = np.flatnonzero(np.asarray(group) == g)
        cnt = off[idx + 1] - off[idx]
        vis = np.concatenate([np.arange(off[k], off[k + 1]) for k in idx]) if cnt.sum() else np.zeros(0, dtype=np.int64)
        sub = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
        N, Bg, z, Kg = misclass_sweep_stats(seed, i, i == 1, n, T[g], Cm[g], theta, y[idx], cens[idx], sub, t[vis], stage[vis],
                                            E, zbits, u=None if u is None else u[idx], pi=pi, obs=idx)
        Ns.append(N); zs.append(z); B = B + Bg; K = K + Kg
    return np.array(Ns), B, np.array(zs), K


def gibbs_misclass(seed, it, n, nu, zeta, T, Cm, y, cens, offsets, t, stage, E, start, zbits, u=None, pi=None, beta=None,
                   alpha=None, group=None):
    """The method-64 chain with stage visits from the host restatement: misclass_sweep_stats + po.update per sweep, with
    beta the Dirichlet update of pi (as pyoracle_panel.gibbs_panel) and with alpha the update of E's rows (Gamma(alpha + K,
    1) draws on parameter sub-streams m + n + c S + o for alpha > 0, each row normalised in index order).  With group
    (group[k] in 0..G-1; T, Cm then (G, (n+1)^2)) every group's observations are drawn on its own structure, theta is
    gathered over the groups as pyoracle_groups.groups_update does, and B and K are summed over the groups.  Returns (theta
    rows (it, m), pi rows (it, n), E rows (it, n, S)), row 0 the start values."""
    y = _f64(y); cens = np.asarray(cens); u = None if u is None else _f64(u)
    theta = _f64(start).copy(); m = theta.shape[0]
    pi = np.eye(n)[0] if pi is None else _f64(pi).copy()
    Em = _f64(E).copy(); Sn = Em.shape[1]
    res = np.zeros((it, m)); res[0] = theta
    pis = np.zeros((it, n)); pis[0] = pi
    Es = np.zeros((it, n, Sn)); Es[0] = Em
    for i in range(1, it):
        if group is None:
            N, B, z, K = misclass_sweep_stats(seed, i, i == 1, n, T, Cm, theta, y, cens, offsets, t, stage, Em, zbits, u=u, pi=pi)
            theta = po.update(seed, i, n, nu, zeta, T, Cm, zbits, N, z)
        else:
            N, B, z, K = _group_stats(seed, i, n, T, Cm, theta, y, cens, offsets, t, stage, Em, zbits, u, pi, group)
            theta = pg.groups_update(seed, i, n, nu, zeta, T, Cm, zbits, N, z)
        if beta is not None:
            g = [po.rgamma_at(seed, i, m + k, float(beta[k]) + float(B[k]), 1.0) for k in range(n)]
            tot = 0.0
            for v in g:
                tot += v
            pi = np.array([v / tot for v in g])
        if alpha is not None:
            a = _f64(alpha)
            Em = np.zeros((n, Sn))
            for c in range(n):
                g = [po.rgamma_at(seed, i, m + n + c * Sn + o, float(a[c, o]) + float(K[c, o]), 1.0) if a[c, o] > 0 else 0.0
                     for o in range(Sn)]
                tot = 0.0
                for v in g:
                    tot += v
                Em[c] = [g[o] / tot if a[c, o] > 0 else 0.0 for o in range(Sn)]
        res[i] = theta; pis[i] = pi; Es[i] = Em
    return res, pis, Es
