"""Delayed entry (left truncation) for the uniformisation sampler in its host build, oracle/pht_oracle_entry.c: the ghost
counts are Geometric(S(a)), the ghost paths have the left-censored law on (0, a], the shared log1p is accurate, and the
augmented chain of a one-phase model has the closed-form truncated-data posterior."""
import numpy as np
import pytest
import scipy.linalg as sl
from scipy import stats

from oracle import pyoracle as po
from oracle import pyoracle_entry as pe
from phasetype_b200 import synth
from tests import util
from tests.test_unif_oracle import GENERATORS, _S, expectations


def _survival(Sm, pi, a):
    return float(pi @ sl.expm(Sm * a) @ np.ones(Sm.shape[0]))


def _case(name):
    if name == "dense8":
        R, s = util.dense_rates(8, np.random.default_rng(88))
        return R, s, np.eye(8)[0]
    if name == "sm_general_pi":
        R, s = GENERATORS["sm"]
        pi = np.array([0.2, 0.5, 0.3])
        return R, s, pi
    R, s = GENERATORS[name]
    return R, s, np.eye(s.shape[0])[0]


CASES = ["erlang4", "tied_coxian", "dense8", "sm_general_pi"]


def test_entry_tables_give_survival_and_failure():
    for name in CASES:
        R, s, pi = _case(name)
        Sm = _S(R, s)
        sig, phi = pe.entry_tables(Sm.ravel(order="F"), s, pi=pi, tmax=3.0)
        lam = -np.diag(Sm).min()
        assert (sig >= 0).all() and (phi >= 0).all()
        for a in (0.2, 1.0, 3.0):
            k = np.arange(pe.pu.truncation(lam * a) + 1)
            w = stats.poisson.pmf(k, lam * a)
            Sa = _survival(Sm, pi, a)
            assert abs(w @ sig[k] - Sa) < 1e-12 and abs(w @ phi[k] - (1 - Sa)) < 1e-12, (name, a)


@pytest.mark.parametrize("name", CASES)
def test_ghost_count_is_geometric(name):
    R, s, pi = _case(name)
    Sm = _S(R, s); S = Sm.ravel(order="F")
    l = 100000
    for j, a0 in enumerate((0.4, 1.5, 3.0)):
        Sa = _survival(Sm, pi, a0)
        a = np.full(l, a0); y = a + 0.25
        cens = np.arange(l, dtype=np.int32) % 2
        M, _, _, _, err = pe.entry_paths(11 + j, 2, y, cens, a, S, s, pi=pi, paths=False)
        assert err == 0
        F = 1.0 - Sa
        mean, sd = F / Sa, np.sqrt(F) / Sa
        assert abs(M.mean() - mean) < 4.5 * sd / np.sqrt(l) + 1e-12, (name, a0, M.mean(), mean)
        # chi-square over k: the bins with at least 20 expected, then the tail
        p = stats.geom.pmf(np.arange(1, 10000), Sa)             # P(M = k - 1)
        kmax = int(np.searchsorted(-(l * p), -20.0))
        if kmax < 1:
            continue
        obs = np.bincount(np.minimum(M, kmax), minlength=kmax + 1)[:kmax + 1]
        exp_ = np.r_[l * p[:kmax], l * (1.0 - p[:kmax].sum())]
        if kmax == 0 or exp_[-1] < 5:
            obs = np.r_[obs[:-2], obs[-2:].sum()]; exp_ = np.r_[exp_[:-2], exp_[-2:].sum()]
        chi2 = ((obs - exp_) ** 2 / exp_).sum()
        assert stats.chi2.sf(chi2, len(obs) - 1) > 1e-4, (name, a0, chi2, len(obs))


def test_no_ghosts_without_truncation():
    R, s, pi = _case("dense8")
    S = _S(R, s).ravel(order="F")
    y = np.random.default_rng(3).exponential(1.0, 2000)
    M, B, N, z, err = pe.entry_paths(5, 1, y, np.zeros(2000, dtype=np.int32), np.zeros(2000), S, s)
    assert err == 0 and (M == 0).all() and B.shape == (0,)


@pytest.mark.parametrize("name", CASES)
def test_ghost_paths_have_the_left_censored_law(name):
    R, s, pi = _case(name)
    Sm = _S(R, s); S = Sm.ravel(order="F"); n = s.shape[0]
    a0 = 1.2
    Sa = _survival(Sm, pi, a0)
    l = int(min(400000, np.ceil(120000 * Sa / (1 - Sa))))
    a = np.full(l, a0)
    M, B, N, z, err = pe.entry_paths(21, 3, a, np.zeros(l, dtype=np.int32), a, S, s, pi=pi)
    assert err == 0
    G = B.shape[0]
    assert G == M.sum() and G > 50000
    Ez, EN, Eexit, EB = expectations(Sm, s, pi, 0.0, "left", a0)
    Nm = N.reshape(G, n, n).transpose(0, 2, 1)
    tol = lambda v: 4.5 * v.std(0) / np.sqrt(G) + 2e-4
    assert (np.abs(z.mean(0) - Ez) < tol(z)).all(), (z.mean(0), Ez)
    off = Nm * (1 - np.eye(n))
    assert (np.abs(off.mean(0) - EN) < tol(off)).all()
    ex = np.diagonal(Nm, axis1=1, axis2=2)
    assert (np.abs(ex.mean(0) - Eexit) < tol(ex)).all(), (ex.mean(0), Eexit)
    Bh = np.bincount(B, minlength=n) / G
    assert (np.abs(Bh - EB) < 4.5 * np.sqrt(np.clip(EB * (1 - EB), 0, None) / G) + 2e-4).all(), (Bh, EB)
    assert (ex.sum(1) == 1).all() and (z.sum(1) <= a0 * (1 + 1e-12)).all() and (z.sum(1) > 0).all()


def test_ghost_count_of_a_hopeless_entry_age_raises_bit_1024():
    R, s = np.zeros((1, 1)), np.array([1.0])
    S = _S(R, s).ravel(order="F")
    a = np.array([30.0, 900.0])
    M, _, _, _, err = pe.entry_paths(1, 1, a, np.zeros(2, dtype=np.int32), a, S, s, paths=False)
    assert err == 1024 and M[1] == 0


def test_log1p_within_one_ulp_and_fast_path_equals_general_path():
    rng = np.random.default_rng(4)
    xs = np.concatenate([rng.uniform(-1, 1, 30000), -rng.uniform(0, 1, 10000) ** 6, rng.uniform(-0.3, 0.42, 20000),
                         np.exp(rng.uniform(-700, 700, 20000)), -np.exp(rng.uniform(-700, -1e-9, 10000)),
                         rng.normal(0, 1e-8, 5000), np.array([0.0, -0.0, 5e-324, -5e-324, 1e300, 2.0 ** 53, 2.0 ** 60,
                                                             np.nextafter(-1.0, 0.0), -0.2928932188134524,
                                                             np.nextafter(-0.2928932188134524, -1), 0.41421356237309503,
                                                             np.nextafter(0.41421356237309503, 0)])])
    xs = xs[xs > -1.0]
    got = np.array([pe.log1p(x) for x in xs]); ref = np.log1p(xs)
    assert (np.abs(got - ref) <= np.spacing(np.abs(ref))).all(), xs[np.abs(got - ref) > np.spacing(np.abs(ref))][:5]
    fast = xs[(xs >= -0.2928932188134524) & (xs < 0.41421356237309503)]
    assert fast.size > 30000
    for x in fast:
        g, h = pe.log1p(x), pe.log1p_general(x)
        assert g == h and np.signbit(g) == np.signbit(h), x
    assert pe.log1p(-1.0) == -np.inf and np.isnan(pe.log1p(-1.5)) and np.isnan(pe.log1p(np.nan)) and pe.log1p(np.inf) == np.inf


def _exponential_data(rate, l, rng):
    """Delayed-entry exponential data: entry ages U(0, 3), a fifth right-censored."""
    R, s = np.zeros((1, 1)), np.array([rate])
    y, a, cens, _ = synth.delayed_entry(R, s, l, lambda k, r: r.uniform(0.0, 3.0, k), rng,
                                        censor=lambda k, r: np.where(r.random(k) < 0.2, r.uniform(0.0, 6.0, k), np.inf))
    return y, a, cens


def _batch_means(x, batches=40):
    b = x.shape[0] // batches
    m = x[:b * batches].reshape(batches, b).mean(1)
    return x.mean(), m.std(ddof=1) / np.sqrt(batches)


def test_exact_posterior_of_the_exponential_model():
    """One phase, Gamma(nu, zeta) prior: the truncated-data posterior is Gamma(nu + d, zeta + sum(y - a)).  The chain
    with entry ages has its mean and variance; the chain that ignores them does not."""
    rng = np.random.default_rng(77)
    y, a, cens = _exponential_data(0.8, 120, rng)
    nu, zeta = np.array([2.0]), np.array([1.5])
    T = np.array([0, 0, 1, 0], dtype=np.int32); Cm = np.ones(4)
    d = int((cens == 0).sum())
    shape, rate = nu[0] + d, zeta[0] + (y - a).sum()
    mean, var = shape / rate, shape / rate ** 2
    zbits = po.choose_zbits(float((y + a).sum()))
    it = 6001
    th = pe.gibbs_entry(5, it, 1, nu, zeta, T, Cm, y, cens, a, np.array([1.0]), zbits)[201:, 0]
    m, se = _batch_means(th)
    assert abs(m - mean) < 4.5 * se, (m, mean, se)
    v, sev = _batch_means((th - mean) ** 2)
    assert abs(v - var) < 4.5 * sev, (v, var, sev)
    # without the entry ages: the same check fails by far
    th0 = pe.gibbs_entry(5, 2001, 1, nu, zeta, T, Cm, y, cens, np.zeros_like(a), np.array([1.0]), zbits)[201:, 0]
    m0, se0 = _batch_means(th0)
    assert abs(m0 - mean) > 10 * max(se, se0), (m0, mean)
