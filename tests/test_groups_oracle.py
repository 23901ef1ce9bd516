"""The host restatement of groups with their own structure (oracle/pht_oracle_groups.c), on the CPU: one group is the
existing method-64 host chain bit for bit, and a two-group exponential model recovers its closed-form posteriors, both
with a parameter per group and with one parameter shared by the groups.  Also the grouped data generator."""
import numpy as np

from oracle import pyoracle as po
from oracle import pyoracle_entry as pe
from oracle import pyoracle_groups as pg
from phasetype_b200 import synth
from tests import util


def test_one_group_is_the_method_64_host_chain():
    rng = np.random.default_rng(11)
    n, l = 4, 400
    R, s = util.dense_rates(n, rng)
    T, Cm, theta = util.general_model(R, s)
    m = theta.shape[0]
    y = rng.exponential(1.0, l) + 0.01
    kind = rng.integers(0, 4, l)
    cens = (kind > 0).astype(np.int32)
    y = np.where(kind == 3, 0.0, y)
    u = np.where(kind >= 2, y + rng.exponential(0.7, l) + 1e-3, np.inf)
    zbits = po.choose_zbits(float(np.where(np.isfinite(u), u, y).sum()))
    nu, zeta = np.full(m, 2.0), np.full(m, 2.0)
    want = pe.gibbs_entry(9, 12, n, nu, zeta, T, Cm, y, cens, np.zeros(l), theta, zbits, u=u)
    got = pg.gibbs_groups(9, 12, n, nu, zeta, np.asarray(T)[None], np.asarray(Cm)[None], y, cens, np.zeros(l, np.int32),
                          theta, zbits, u=u)
    assert np.array_equal(got, want)


def _exp_data(rng, rates, sizes):
    T = np.array([[0, 0, 1, 0], [0, 0, 2, 0]], dtype=np.int32)
    y, cens, group = synth.groups(T, np.ones((2, 4)), rates, 1, sizes, rng, censor=lambda k, r: r.uniform(0.0, 2.0, k))
    return y, cens, group


def _check(draws, shape, rate):
    mean, var = shape / rate, shape / rate ** 2
    se = np.sqrt(var / draws.size)                  # n = 1: the statistics are the data, so the draws are independent
    assert abs(draws.mean() - mean) < 5.0 * se, (draws.mean(), mean, se)
    assert abs(draws.var() / var - 1.0) < 0.1, (draws.var(), var)


def test_two_group_exponential_posteriors():
    """Group g exits at theta_g: theta_g ~ Gamma(nu + d_g, zeta + sum y_g); both mapped to theta_1: Gamma(nu + d_0 + d_1,
    zeta + sum y)."""
    rng = np.random.default_rng(5)
    y, cens, group = _exp_data(rng, np.array([0.7, 2.5]), (300, 500))
    nu, zeta = 2.0, 1.0
    zbits = po.choose_zbits(float(y.sum()))
    d = [int(((cens == 0) & (group == g)).sum()) for g in (0, 1)]
    sy = [float(y[group == g].sum()) for g in (0, 1)]
    it = 3001
    T = np.array([[0, 0, 1, 0], [0, 0, 2, 0]], dtype=np.int32)
    th = pg.gibbs_groups(3, it, 1, [nu, nu], [zeta, zeta], T, np.ones((2, 4)), y, cens, group, np.array([1.0, 1.0]), zbits)[1:]
    for g in (0, 1):
        _check(th[:, g], nu + d[g], zeta + sy[g])
    shared = np.array([[0, 0, 1, 0], [0, 0, 1, 0]], dtype=np.int32)
    th1 = pg.gibbs_groups(3, it, 1, [nu], [zeta], shared, np.ones((2, 4)), y, cens, group, np.array([1.0]), zbits)[1:, 0]
    _check(th1, nu + d[0] + d[1], zeta + sy[0] + sy[1])


def test_group_stats_sum_to_the_single_structure_stats_for_one_structure():
    """Two groups with the same structure: the per-group statistics add up to those of one group holding every observation."""
    rng = np.random.default_rng(8)
    n, l = 3, 300
    R, s = util.dense_rates(n, rng)
    T, Cm, theta = util.general_model(R, s)
    y = rng.exponential(1.0, l) + 0.01
    cens = (rng.random(l) < 0.3).astype(np.int32)
    group = rng.integers(0, 2, l).astype(np.int32)
    zbits = po.choose_zbits(float(y.sum()))
    TT, CC = np.stack([T, T]), np.stack([Cm, Cm])
    N, B, z = pg.groups_sweep_stats(4, 3, False, n, TT, CC, theta, y, cens, group, zbits)
    N1, B1, z1 = pg.groups_sweep_stats(4, 3, False, n, np.asarray(T)[None], np.asarray(Cm)[None], theta, y, cens,
                                       np.zeros(l, np.int32), zbits)
    assert np.array_equal(N.sum(0), N1[0]) and np.array_equal(B.sum(0), B1[0]) and np.array_equal(z.sum(0), z1[0])
    assert B[0].sum() == (group == 0).sum() and B[1].sum() == (group == 1).sum()


def test_synth_groups_uses_each_groups_generator():
    rng = np.random.default_rng(2)
    T = np.array([[0, 0, 1, 0], [0, 0, 2, 0]], dtype=np.int32)
    y, cens, group = synth.groups(T, np.ones((2, 4)), np.array([0.5, 4.0]), 1, (20000, 30000), rng)
    assert y.shape == (50000,) and not cens.any()
    assert np.array_equal(group, np.repeat([0, 1], [20000, 30000]))
    assert abs(y[group == 0].mean() - 2.0) < 0.05 and abs(y[group == 1].mean() - 0.25) < 0.005
