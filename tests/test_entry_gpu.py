"""Delayed entry (left truncation) on the device (method 64, k_unif.cu): ghost counts and ghost paths bit for bit against
the host build (oracle/pht_oracle_entry.c), the observations' own paths untouched, a = 0 equal to no entry ages, sweep
statistics and chains, several GPUs, the closed-form posterior of the exponential model, recovery of rates from
delayed-entry data, and the refusals."""
import threading

import numpy as np
import pytest

from oracle import pyoracle_entry as pe
from phasetype_b200 import synth
from phasetype_b200._lib import METHOD_UNIF
from tests import util

pytestmark = pytest.mark.gpu


def _mixed_entry(n, l, rng):
    """Dense n-phase model; a third each of exact, right- and interval-censored observations, 60 % with an entry age in
    (0, y]."""
    R, s = util.dense_rates(n, rng)
    y = rng.exponential(1.0, l) + 0.01
    kind = rng.integers(0, 3, l)
    cens = (kind > 0).astype(np.int32)
    u = np.where(kind == 2, y + rng.exponential(0.7, l) + 1e-3, np.inf)
    a = np.where(rng.random(l) < 0.6, y * rng.random(l), 0.0)
    return R, s, y, cens, u, a


def _sum_zbits(y, u, a):
    return float((np.where(np.isfinite(u), u, y) + a).sum())


def _engine(R, s, y, cens, u=None, a=None, seed=7, **kw):
    import phasetype_b200 as pb
    n = s.shape[0]
    T, C, theta = util.general_model(R, s)
    m = theta.shape[0]
    uu = np.full(y.shape[0], np.inf) if u is None else u
    aa = np.zeros(y.shape[0]) if a is None else a
    eng = pb.Engine(n, T, C, np.full(m, 2.0), np.full(m, 2.0), y, cens, method=METHOD_UNIF, seed=seed,
                    sum_y_global=_sum_zbits(y, uu, aa), **kw)
    if u is not None:
        eng.set_upper(u)
    if a is not None:
        eng.set_entry(a)
    return eng, T, C, theta


# the most lanes k_unif_ghosts can hold resident on a B200: 148 SMs x 2048 threads, whatever its occupancy
MAX_RESIDENT_LANES = 148 * 2048


@pytest.mark.parametrize("n,l,general_pi", [(1, 2000000, False), (3, 1500000, True), (8, 1000000, False), (8, 1200000, True),
                                            (16, 20000, False), (32, 6000, True)])
def test_ghosts_match_oracle(n, l, general_pi):
    """Ghost counts and every ghost path (B, N, z) bit for bit; for n <= 8 the shards give more ghosts than the device can
    hold resident lanes, so that warps take further chunks of the flat ghost list."""
    rng = np.random.default_rng(300 + n)
    R, s, y, cens, u, a = _mixed_entry(n, l, rng)
    eng, _, _, theta = _engine(R, s, y, cens, u, a, seed=0xE17)
    pi = None
    if general_pi:
        pi = rng.uniform(0.1, 1.0, n); pi /= pi.sum()
        eng.set_pi(pi)
    eng.set_theta(theta, next_iter=4)
    M, B, N, z = eng.entry_paths()
    mdl = eng.model()
    eng.close()
    Mo, Bo, No, zo, err = pe.entry_paths(0xE17, 4, y, cens, a, mdl["S"], mdl["s"], u=u, pi=pi)
    assert err == 0
    assert M.sum() > (MAX_RESIDENT_LANES if n <= 8 else 1000)
    assert np.array_equal(M, Mo)
    assert np.array_equal(B, Bo) and np.array_equal(N, No) and np.array_equal(z, zo)


def test_window_in_the_middle_of_the_shard():
    rng = np.random.default_rng(5)
    R, s, y, cens, u, a = _mixed_entry(6, 30000, rng)
    eng, _, _, theta = _engine(R, s, y, cens, u, a, seed=99)
    eng.set_theta(theta, next_iter=2)
    M, B, N, z = eng.entry_paths(12345, 7000)
    mdl = eng.model()
    eng.close()
    Mo, Bo, No, zo, err = pe.entry_paths(99, 2, y[12345:19345], cens[12345:19345], a[12345:19345], mdl["S"], mdl["s"],
                                         u=u[12345:19345], obs0=12345)
    assert err == 0 and np.array_equal(M, Mo) and np.array_equal(B, Bo) and np.array_equal(N, No) and np.array_equal(z, zo)


def test_observed_paths_unchanged_by_entry_ages():
    rng = np.random.default_rng(6)
    R, s, y, cens, u, a = _mixed_entry(8, 50000, rng)
    eng, _, _, theta = _engine(R, s, y, cens, u, a, seed=3)
    eng.set_theta(theta, next_iter=5)
    with_a = eng.paths()
    eng.set_entry(None)
    without = eng.paths()
    eng.close()
    for x, w in zip(with_a, without):
        assert np.array_equal(x, w)


def test_zero_entry_ages_give_the_chain_without_them():
    rng = np.random.default_rng(7)
    R, s, y, cens, u, a = _mixed_entry(5, 20000, rng)
    import phasetype_b200 as pb
    zbits = pb.lib().pht_choose_zbits(_sum_zbits(y, u, a))       # room for the truncated run below
    plain, _, _, theta = _engine(R, s, y, cens, u, seed=21, zbits=zbits)
    eng, _, _, _ = _engine(R, s, y, cens, u, seed=21, zbits=zbits)
    plain.set_theta(theta, 1)
    want = plain.run(8)
    plain.close()
    eng.set_entry(np.zeros(y.shape[0]))
    eng.set_theta(theta, 1)
    assert np.array_equal(eng.run(8), want)
    eng.set_entry(a)                        # a truncated run in between
    eng.set_theta(theta, 1)
    trunc = eng.run(8)
    assert not np.array_equal(trunc, want)
    eng.set_entry(None)
    eng.set_theta(theta, 1)
    assert np.array_equal(eng.run(8), want)
    eng.close()


def test_sweep_stats_c3_with_entry_match_oracle():
    """10^6 observations of the C3 shape (20 % right-censored) with entry ages, in the production layout."""
    import phasetype_b200 as pb
    wl = synth.config(3, "MHRS", l=10 ** 6)
    rng = np.random.default_rng(9)
    a = np.where(rng.random(wl.l) < 0.5, wl.y * rng.random(wl.l), 0.0)
    eng = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=METHOD_UNIF, seed=2718,
                    sum_y_global=float((wl.y + a).sum()))
    eng.set_entry(a)
    eng.set_theta(wl.theta, next_iter=3)
    N, B, z = eng.sweep_stats()
    zbits = eng.zbits
    eng.close()
    No, Bo, zo = pe.entry_sweep_stats(2718, 3, True, wl.n, wl.T, wl.C, wl.theta, wl.y, wl.censored, a, zbits)
    assert np.array_equal(N, No) and np.array_equal(B, Bo) and np.array_equal(z, zo)


def _chain_workload(l=20000):
    rng = np.random.default_rng(12)
    R, s, y, cens, u, a = _mixed_entry(5, l, rng)
    T, C, theta = util.general_model(R, s)
    return R, s, y, cens, u, a, T, C, theta


def test_chain_equals_oracle():
    import phasetype_b200 as pb
    R, s, y, cens, u, a, T, C, theta = _chain_workload()
    m = theta.shape[0]
    eng = pb.Engine(5, T, C, np.full(m, 2.0), np.full(m, 2.0), y, cens, method=METHOD_UNIF, seed=31,
                    sum_y_global=_sum_zbits(y, u, a))
    eng.set_upper(u)
    eng.set_entry(a)
    eng.set_theta(theta, next_iter=1)
    got = eng.run(20)
    zbits = eng.zbits
    eng.close()
    want = pe.gibbs_entry(31, 21, 5, np.full(m, 2.0), np.full(m, 2.0), T, C, y, cens, a, theta, zbits, u=u)
    assert np.array_equal(got, want[1:])


def test_two_gpus_equal_one():
    import phasetype_b200 as pb
    if pb.lib().pht_device_count() < 2:
        pytest.skip("needs two or more GPUs")
    R, s, y, cens, u, a, T, C, theta = _chain_workload(40000)
    m = theta.shape[0]
    sy = _sum_zbits(y, u, a)

    def engine(rank, world):
        e = pb.Engine(5, T, C, np.full(m, 2.0), np.full(m, 2.0), y[rank::world], cens[rank::world], method=METHOD_UNIF, seed=8,
                      device=rank, rank=rank, world=world, use_graph=False, sum_y_global=sy)
        e.set_upper(u[rank::world])
        e.set_entry(a[rank::world])
        return e
    one = engine(0, 1)
    one.set_theta(theta, 1)
    want = one.run(6)
    one.close()
    engs = [engine(r, 2) for r in range(2)]
    handles = b"".join(e.peer_handle() for e in engs)
    for e in engs:
        e.peer_attach(handles)
        e.set_theta(theta, 1)
    outs = [None, None]

    def work(r):
        outs[r] = engs[r].run(6)
    th = [threading.Thread(target=work, args=(r,)) for r in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    for e in engs:
        e.close()
    assert np.array_equal(outs[0], want) and np.array_equal(outs[1], want)


def _batch_means(x, batches=40):
    b = x.shape[0] // batches
    mb = x[:b * batches].reshape(batches, b).mean(1)
    return x.mean(), mb.std(ddof=1) / np.sqrt(batches)


def test_exact_posterior_of_the_exponential_model():
    """One phase, Gamma(nu, zeta) prior, truncated exact and right-censored data: Gamma(nu + d, zeta + sum(y - a))."""
    import phasetype_b200 as pb
    rng = np.random.default_rng(78)
    R, s = np.zeros((1, 1)), np.array([0.8])
    y, a, cens, _ = synth.delayed_entry(R, s, 150, lambda k, r: r.uniform(0.0, 3.0, k), rng,
                                        censor=lambda k, r: np.where(r.random(k) < 0.2, r.uniform(0.0, 6.0, k), np.inf))
    T = np.array([0, 0, 1, 0], dtype=np.int32)
    eng = pb.Engine(1, T, np.ones(4), [2.0], [1.5], y, cens, method=METHOD_UNIF, seed=17, sum_y_global=float((y + a).sum()))
    eng.set_entry(a)
    eng.set_theta(np.array([1.0]), 1)
    th = eng.run(20000)[500:, 0]
    eng.close()
    d = int((cens == 0).sum())
    shape, rate = 2.0 + d, 1.5 + (y - a).sum()
    m, se = _batch_means(th)
    assert abs(m - shape / rate) < 4.5 * se, (m, shape / rate, se)
    v, sev = _batch_means((th - shape / rate) ** 2)
    assert abs(v - shape / rate ** 2) < 4.5 * sev, (v, shape / rate ** 2, sev)


def test_rates_recovered_from_delayed_entry_data():
    """Units of the tied 4-phase Coxian (forward rate F, early exit R; test_unif_gpu) enter at ages U(0, 3), so many are
    lost before entry; the posterior means land within 10 % of the truth with the entry ages, and clearly off without."""
    import phasetype_b200 as pb
    from tests.test_unif_gpu import _tied_model
    F, Rx = 1.5, 0.3
    R = np.diag(np.full(3, F), 1); s = np.array([Rx, Rx, Rx, F])
    truth = np.array([F, Rx])
    rng = np.random.default_rng(404)
    y, a = synth.delayed_entry(R, s, 30000, lambda k, r: r.uniform(0.0, 3.0, k), rng)
    T, C = _tied_model()
    cens = np.zeros(y.shape[0], dtype=np.int32)
    means = []
    for with_entry in (True, False):
        eng = pb.Engine(4, T, C, np.ones(2), np.ones(2), y, cens, method=METHOD_UNIF, seed=5,
                        sum_y_global=float((y + a).sum()))
        if with_entry:
            eng.set_entry(a)
        eng.set_theta(np.ones(2), next_iter=1)
        means.append(eng.run(400)[150:].mean(0))
        eng.close()
    err_with = np.abs(means[0] / truth - 1.0)
    err_without = np.abs(means[1] / truth - 1.0)
    assert (err_with < 0.1).all(), means[0]
    assert err_without.max() > 0.2 and err_without.max() > 2 * err_with.max(), (means[1], means[0])


@pytest.mark.parametrize("case,msg", [("nan", "must be finite"), ("inf", "must be finite"), ("negative", "is negative"),
                                      ("above", "above y"), ("left", "above y"), ("zbits", "too fine")])
def test_bad_entry_ages_are_refused(case, msg):
    import phasetype_b200 as pb
    rng = np.random.default_rng(9)
    R, s = util.dense_rates(3, rng)
    y = rng.exponential(1.0, 50) + 0.01
    cens = np.ones(50, dtype=np.int32); cens[:5] = 0
    u = np.full(50, np.inf); u[20:40] = y[20:40] + 1.0
    y[45] = 0.0; u[45] = 0.5                 # a left-censored record
    a = 0.5 * y
    if case == "nan":
        a[30] = np.nan
    elif case == "inf":
        a[30] = -np.inf
    elif case == "negative":
        a[30] = -0.1
    elif case == "above":
        a[10] = y[10] + 0.01
    elif case == "left":
        a[45] = 0.1
    if case == "zbits":
        # sum y = 40 allows 52 fractional bits, sum (y + a) = 79.96 only 51
        y = np.ones(40); cens = np.zeros(40, dtype=np.int32); u = None; a = 0.999 * y
    eng, _, _, _ = _engine(R, s, y, cens, u)
    if case == "zbits":
        assert eng.zbits == 52
    with pytest.raises(pb.EngineError, match=msg):
        eng.set_entry(a)
    eng.close()


def test_entry_ages_refused_after_attach():
    import phasetype_b200 as pb
    if pb.lib().pht_device_count() < 2:
        pytest.skip("needs two or more GPUs")
    R, s = util.dense_rates(3, np.random.default_rng(2))
    y = np.ones(10); cens = np.zeros(10, dtype=np.int32)
    T, C, theta = util.general_model(R, s)
    m = theta.shape[0]
    engs = [pb.Engine(3, T, C, np.ones(m), np.ones(m), y[r::2], cens[r::2], method=METHOD_UNIF, device=r, rank=r, world=2,
                      sum_y_global=20.0) for r in range(2)]
    h = b"".join(e.peer_handle() for e in engs)
    for e in engs:
        e.peer_attach(h)
    with pytest.raises(pb.EngineError, match="before the exchange windows"):
        engs[0].set_entry(np.zeros(5))
    for e in engs:
        e.close()


@pytest.mark.parametrize("method", [1, 2, 4, 8, 16])
def test_other_methods_refuse_entry_ages(method):
    import phasetype_b200 as pb
    R, s = util.dense_rates(3, np.random.default_rng(1), symmetric=True)
    T, C, theta = util.general_model(R, s)
    m = theta.shape[0]
    y = np.ones(8); cens = np.zeros(8, dtype=np.int32)
    eng = pb.Engine(3, T, C, np.ones(m), np.ones(m), y, cens, method=method)
    with pytest.raises(pb.EngineError, match="needs method 64"):
        eng.set_entry(np.zeros(8))
    eng.close()


def test_hopeless_entry_age_raises_bit_1024():
    import phasetype_b200 as pb
    y = np.array([1.0, 25.5, 2.0]); a = np.array([0.5, 25.0, 0.0])      # S(25) = 1.4e-11: M would exceed 2^20
    T = np.array([0, 0, 1, 0], dtype=np.int32)
    eng = pb.Engine(1, T, np.ones(4), [2.0], [2.0], y, np.zeros(3, dtype=np.int32), method=METHOD_UNIF, seed=1,
                    sum_y_global=float((y + a).sum()))
    eng.set_entry(a)
    eng.set_theta(np.array([1.0]), 1)
    with pytest.raises(pb.EngineError, match="0x400.*no survival at an observation's entry age"):
        eng.run(1)
    eng.close()
