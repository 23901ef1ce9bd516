"""The uniformisation sampler (method 64) in its host build, oracle/pht_oracle_unif.c: the table reproduces e^{Sy}, the
Poisson truncation stays below its documented bound, and the paths have the exact conditional law (tier 2) for exact,
right-, interval- and left-censored observations and for a start distribution with several positive entries -- on
generators the spectral samplers cannot carry (a Jordan block, a complex spectrum) too."""
import math

import numpy as np
import pytest
import scipy.linalg as sl
from scipy import stats

from oracle import pyoracle_unif as pu
from tests import util

ERLANG4 = (np.diag(np.full(3, 2.0), 1), np.array([0.0, 0.0, 0.0, 2.0]))
ERLANG16 = (np.diag(np.full(15, 3.0), 1), np.r_[np.zeros(15), 3.0])
R4 = np.array([[0.0, 2.6, 0.1, 0.2], [0.15, 0.0, 2.9, 0.1], [0.2, 0.1, 0.0, 2.4], [2.2, 0.2, 0.1, 0.0]])
S4 = np.array([0.5, 0.2, 0.9, 0.3])


def _tied_coxian():
    """S = diag(-1.8, -1.8, -1.8, -1.5) + superdiag(1.5): three phases share forward rate 1.5 and exit rate 0.3."""
    R = np.diag(np.full(3, 1.5), 1)
    return R, np.array([0.3, 0.3, 0.3, 1.5])


def _sm():
    """SURVEY 8(c), unequal exits."""
    Sm = np.array([[-4.1, 1.8, 1.8], [9.5, -11.3, 0.0], [9.5, 0.0, -15.5]])
    R = Sm.copy(); np.fill_diagonal(R, 0.0)
    return R, -Sm.sum(1)


def _stiff():
    R = np.array([[0.0, 400.0, 0.0], [0.05, 0.0, 0.1], [0.0, 900.0, 0.0]])
    return R, np.array([1.0, 0.02, 3.0])


GENERATORS = {"erlang4": ERLANG4, "erlang16": ERLANG16, "tied_coxian": _tied_coxian(), "complex_r4": (R4, S4), "sm": _sm(),
              "dense32": util.dense_rates(32, np.random.default_rng(32)), "stiff": _stiff()}


def _S(R, s):
    S = R.copy()
    np.fill_diagonal(S, -(R.sum(1) + s))
    return S


@pytest.mark.parametrize("name", sorted(GENERATORS))
def test_table_reproduces_expm(name):
    R, s = GENERATORS[name]
    Sm = _S(R, s); n = s.shape[0]
    for y in (0.05, 1.0, 2.5):
        K, t = pu.table(Sm.ravel(order="F"), s, tmax=y)
        assert K >= 0
        x = t["lam"] * y
        k = np.arange(pu.truncation(x) + 1)
        w = stats.poisson.pmf(k, x)
        E = np.einsum("k,kij->ij", w, t["P"][:k.shape[0]])
        X = sl.expm(Sm * y)
        assert np.abs(E - X).max() <= 1e-12 * np.abs(X).max(), (name, y)
        # the absorbing column: g_k = 1 - R^k 1, built from non-negative terms only
        g = t["g"][:k.shape[0]]
        assert np.allclose(g, 1.0 - t["P"][:k.shape[0]].sum(2), rtol=0, atol=1e-10)
        assert (g >= 0).all()
    # log k! of the table against lgamma
    assert np.allclose(t["lgk"][1:2000], [math.lgamma(k + 1) for k in range(1, 2000)], rtol=1e-12, atol=1e-13)


def test_truncation_tail_below_bound():
    """P(Pois(x) > K(x)) < 1e-15 for every x the table admits (K(x) < 4096)."""
    xs = np.concatenate([np.linspace(0.0, 10.0, 2001), np.linspace(10.0, 3484.0, 4000)])
    Ks = np.array([pu.truncation(x) for x in xs])
    assert Ks.max() < pu.CAP
    tail = stats.poisson.sf(Ks, xs)
    assert tail.max() < 1e-15, (xs[tail.argmax()], tail.max())
    assert pu.truncation(3600.0) >= pu.CAP                 # beyond: error bit 256, not a silent truncation


def _num(Sm, s, pi, t):
    """E[X; T > t] for the path statistics X: (z, N off-diagonal, exits, start state), with their normaliser P(T > t)."""
    n = s.shape[0]
    one = np.ones(n)
    et = sl.expm(Sm * t)
    post = pi @ et @ np.linalg.inv(-Sm)
    I = np.zeros((n, n))
    for i in range(n):
        for j in range(n):
            if i != j and Sm[i, j] == 0.0:
                continue
            E = np.zeros((n, n)); E[i, j] = 1.0
            A = np.block([[Sm, E], [np.zeros((n, n)), Sm]])
            I[i, j] = pi @ sl.expm(A * t)[:n, n:] @ one if t > 0 else 0.0
    z = np.diag(I) + post
    N = (I + post[:, None]) * Sm * (1 - np.eye(n))
    return z, N, post * s, pi * (et @ one), pi @ et @ one


def expectations(Sm, s, pi, y, kind, u=None):
    """E[z], E[N_ij] (i != j), E[exits from b], P(start = a) of a path given the observation (kind exact / right /
    interval / left), for a general start distribution pi (Van Loan block integrals)."""
    n = s.shape[0]
    if kind == "exact":
        ey = sl.expm(Sm * y); f = pi @ ey @ s
        I = np.zeros((n, n))
        for i in range(n):
            for j in range(n):
                if i != j and Sm[i, j] == 0.0:
                    continue
                E = np.zeros((n, n)); E[i, j] = 1.0
                A = np.block([[Sm, E], [np.zeros((n, n)), Sm]])
                I[i, j] = pi @ sl.expm(A * y)[:n, n:] @ s / f
        return np.diag(I).copy(), I * Sm * (1 - np.eye(n)), (pi @ ey) * s / f, pi * (ey @ s) / f
    a = _num(Sm, s, pi, y)
    if kind == "right":
        return tuple(v / a[4] for v in a[:4])
    b = _num(Sm, s, pi, u)
    return tuple((va - vb) / (a[4] - b[4]) for va, vb in zip(a[:4], b[:4]))


def _check(Sm, s, pi, y0, kind, u0=None, l=200000, seed=5):
    n = s.shape[0]
    y = np.full(l, y0); cens = np.full(l, 0 if kind == "exact" else 1, dtype=np.int32)
    u = None if u0 is None else np.full(l, u0)
    B, N, z, err = pu.unif_paths(seed, 3, y, cens, Sm.ravel(order="F"), s, u=u, pi=pi)
    assert err == 0
    Ez, EN, Eexit, EB = expectations(Sm, s, pi, y0, kind, u0)
    Nm = N.reshape(l, n, n).transpose(0, 2, 1)          # N[k, i, j] = transitions i -> j of path k (exits on i == i)
    tol = lambda a: 4.5 * a.std(0) / np.sqrt(l) + 2e-4
    assert (np.abs(z.mean(0) - Ez) < tol(z)).all(), (z.mean(0), Ez)
    off = Nm * (1 - np.eye(n))
    assert (np.abs(off.mean(0) - EN) < tol(off)).all()
    ex = np.diagonal(Nm, axis1=1, axis2=2)
    assert (np.abs(ex.mean(0) - Eexit) < tol(ex)).all(), (ex.mean(0), Eexit)
    Bh = np.bincount(B, minlength=n) / l
    assert (np.abs(Bh - EB) < 4.5 * np.sqrt(np.clip(EB * (1 - EB), 0, None) / l) + 2e-4).all(), (Bh, EB)
    assert (ex.sum(1) == 1).all()                       # every path ends in exactly one absorption
    tot = z.sum(1)
    if kind == "exact":
        assert np.allclose(tot, y0, rtol=1e-12)
    elif kind == "right":
        assert (tot >= y0 * (1 - 1e-12)).all()
    else:
        assert (tot >= y0 * (1 - 1e-12)).all() and (tot <= u0 * (1 + 1e-12)).all()


TIER2 = ["erlang4", "tied_coxian", "complex_r4", "sm"]


@pytest.mark.parametrize("name", TIER2)
@pytest.mark.parametrize("kind", ["exact", "right", "interval", "left"])
def test_tier2_conditional_law(name, kind):
    R, s = GENERATORS[name]
    Sm = _S(R, s); n = s.shape[0]
    pi = np.eye(n)[0]
    y0, u0 = {"exact": (1.5, None), "right": (1.5, None), "interval": (1.0, 1.6), "left": (0.0, 0.7)}[kind]
    _check(Sm, s, pi, y0, kind, u0)


@pytest.mark.parametrize("name", ["sm", "complex_r4", "tied_coxian"])
@pytest.mark.parametrize("kind", ["exact", "right", "interval"])
def test_tier2_general_start_distribution(name, kind):
    R, s = GENERATORS[name]
    Sm = _S(R, s); n = s.shape[0]
    pi = np.linspace(1.0, 2.0, n); pi /= pi.sum()
    y0, u0 = {"exact": (0.8, None), "right": (0.8, None), "interval": (0.5, 1.3)}[kind]
    _check(Sm, s, pi, y0, kind, u0)


def test_tier2_dense32_and_stiff():
    for name, y0 in (("dense32", 0.3), ("stiff", 1.0)):
        R, s = GENERATORS[name]
        Sm = _S(R, s)
        _check(Sm, s, np.eye(s.shape[0])[0], y0, "right", l=50000)


def test_infinite_bounds_are_the_right_censored_paths():
    rng = np.random.default_rng(3)
    R, s = util.dense_rates(6, rng)
    S = _S(R, s).ravel(order="F")
    y = rng.exponential(1.0, 3000) + 0.01
    cens = (rng.uniform(size=3000) < 0.6).astype(np.int32)
    pi = rng.uniform(size=6); pi /= pi.sum()
    for p in (None, pi):
        a = pu.unif_paths(9, 2, y, cens, S, s, pi=p)
        b = pu.unif_paths(9, 2, y, cens, S, s, u=np.full(3000, np.inf), pi=p)
        for x, w in zip(a, b):
            assert np.array_equal(x, w)


def test_table_overflow_is_reported():
    R, s = _stiff()
    S = _S(R, s).ravel(order="F")
    B, N, z, err = pu.unif_paths(1, 1, np.array([1.0, 10.0]), np.zeros(2, dtype=np.int32), S, s)
    assert err == 256
