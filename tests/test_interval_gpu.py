"""Interval-censored observations (pht_engine_set_upper, method MHRS): the absorption time is known to lie in [y, u].
Per-observation parity with the CPU restatement (oracle/pht_oracle_iv.c), the u = +inf case against today's engine,
the chain on one and on two GPUs, recovery of the rates from inspection data, and the refusals."""
import threading

import numpy as np
import pytest

from oracle import pyoracle_iv as poi
from phasetype_b200 import synth
from tests import util

pytestmark = pytest.mark.gpu


def _mixed(n, l, rng, narrow=False):
    """Dense n-phase model; a third each of exact, right-censored and interval-censored observations."""
    R, s = util.dense_rates(n, rng)
    y = rng.exponential(1.2, l) + 0.01
    kind = rng.integers(0, 3, l)                        # 0 exact, 1 right-censored, 2 interval
    cens = (kind > 0).astype(np.int32)
    width = rng.uniform(1e-3, 3e-3, l) if narrow else rng.exponential(1.0, l) + 1e-3
    u = np.where(kind == 2, y + width, np.inf)
    return R, s, y, cens, u


def _sum_max(y, u):
    return float(np.where(np.isfinite(u), u, y).sum())


def _engine(R, s, y, cens, u, mhit, seed, cap, **kw):
    import phasetype_b200 as pb
    n = s.shape[0]
    T, C, theta = util.general_model(R, s)
    m = theta.shape[0]
    eng = pb.Engine(n, T, C, np.full(m, 2.0), np.full(m, 2.0), y, cens, method=1, mhit=mhit, seed=seed, mhrs_cap=cap,
                    sum_y_global=_sum_max(y, u), **kw)
    if u is not None:
        eng.set_upper(u)
    return eng, T, C, theta


@pytest.mark.parametrize("n,mhit,cap,narrow", [(4, 1, 0, False), (4, 3, 16, False), (12, 1, 16, False), (12, 3, 0, False),
                                               (24, 1, 0, False), (24, 3, 16, False), (4, 1, 16, False), (12, 1, 0, False),
                                               (24, 3, 0, False), (8, 1, 16, True)])
def test_paths_match_oracle(n, mhit, cap, narrow):
    rng = np.random.default_rng(300 + n + 10 * mhit + cap)
    l = 2000 if narrow else 3000
    R, s, y, cens, u = _mixed(n, l, rng, narrow)
    eng, _, _, theta = _engine(R, s, y, cens, u, mhit, seed=0x1A7E5, cap=cap)
    eng.set_theta(theta, next_iter=5)
    B, N, z = eng.paths()
    mdl = eng.model()
    cnt = eng.counters()
    eng.close()
    Bo, No, zo, co = poi.mhrs_paths_iv(0x1A7E5, 5, y, cens, u, mdl["S"], mdl["s"], mhit=mhit)
    assert np.array_equal(B, Bo)
    assert np.array_equal(N, No)
    assert np.array_equal(z, zo)
    iv = np.isfinite(u)
    tot = z.sum(1)
    # every interval path is absorbed inside its interval (z sums its sojourns in another order than the clock: 1e-12)
    assert (tot[iv] >= y[iv] * (1 - 1e-12)).all() and (tot[iv] <= u[iv] * (1 + 1e-12)).all()
    if cap:
        assert cnt["deferred"] > 0
    if narrow:
        assert cnt["tail_rounds"] >= 4


def test_sweep_stats_in_the_sorted_layout_match_oracle():
    """The production layout (observations by decreasing y, bounds gathered through the permutation) and the default cap."""
    rng = np.random.default_rng(41)
    R, s, y, cens, u = _mixed(8, 100000, rng)
    eng, T, C, theta = _engine(R, s, y, cens, u, 1, seed=77, cap=0)
    eng.set_theta(theta, next_iter=2)
    N, B, z = eng.sweep_stats()
    zbits = eng.zbits
    eng.close()
    No, Bo, zo, _ = poi.sweep_stats_iv(77, 2, True, 1, 8, T, C, theta, y, cens, u, zbits)
    assert np.array_equal(N, No) and np.array_equal(B, Bo) and np.array_equal(z, zo)


def test_infinite_bounds_are_todays_chain():
    wl = synth.config(3, "MHRS", l=20000)
    chains = []
    for bounded in (False, True):
        import phasetype_b200 as pb
        eng = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=1, mhit=1, seed=2024, mhrs_cap=16)
        if bounded:
            eng.set_upper(np.full(wl.l, np.inf))
        eng.set_theta(wl.theta, next_iter=1)
        chains.append(eng.run(5))
        eng.close()
    assert np.array_equal(chains[0], chains[1])


def _interval_workload(l):
    rng = np.random.default_rng(5)
    R, s, y, cens, u = _mixed(6, l, rng, narrow=True)
    T, C, theta = util.general_model(R, s)
    return R, s, y, cens, u, T, C, theta


def test_chain_equals_oracle():
    import phasetype_b200 as pb
    R, s, y, cens, u, T, C, theta = _interval_workload(6000)
    m = theta.shape[0]
    eng = pb.Engine(6, T, C, np.full(m, 2.0), np.full(m, 2.0), y, cens, method=1, mhit=2, seed=31, mhrs_cap=16,
                    sum_y_global=_sum_max(y, u))
    eng.set_upper(u)
    eng.set_theta(theta, next_iter=1)
    got = eng.run(5)
    zbits = eng.zbits
    eng.close()
    want = poi.gibbs_iv(31, 6, 2, 6, np.full(m, 2.0), np.full(m, 2.0), T, C, y, cens, u, theta, zbits)
    assert np.array_equal(got, want[1:])


def test_two_gpus_equal_one(monkeypatch):
    """In-process fan-out over two devices with the exchange windows attached; the global tail from its first round on."""
    import phasetype_b200 as pb
    if pb.lib().pht_device_count() < 2:
        pytest.skip("needs two or more GPUs")
    monkeypatch.setenv("PHT_B200_KSWITCH", "512")
    R, s, y, cens, u, T, C, theta = _interval_workload(20000)
    m = theta.shape[0]
    sy = _sum_max(y, u)

    def engine(rank, world):
        e = pb.Engine(6, T, C, np.full(m, 2.0), np.full(m, 2.0), y[rank::world], cens[rank::world], method=1, mhit=1, seed=8,
                      device=rank, rank=rank, world=world, mhrs_cap=8, use_graph=False, sum_y_global=sy)
        e.set_upper(u[rank::world])
        return e
    one = engine(0, 1)
    one.set_theta(theta, 1)
    want = one.run(5)
    one.close()
    engs = [engine(r, 2) for r in range(2)]
    handles = b"".join(e.peer_handle() for e in engs)
    for e in engs:
        e.peer_attach(handles)
        e.set_theta(theta, 1)
    outs = [None, None]

    def work(r):
        outs[r] = engs[r].run(5)
    th = [threading.Thread(target=work, args=(r,)) for r in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    glob = sum(e.counters()["global_rounds"] for e in engs)
    for e in engs:
        e.close()
    assert np.array_equal(outs[0], want) and np.array_equal(outs[1], want)
    assert glob > 0


def test_inspection_data_recover_the_rates():
    """Tier 3.  Two-phase model with an early exit: state 0 leaves at a to state 1 and at c to absorption, state 1 is
    absorbed at a (distribution determined by (a, c): poles a + c > a).  4000 units inspected every 0.5 up to 4;
    vague Gamma(1, 1) priors.  With the intervals the posterior mean is within 10 % of (a, c) = (1.2, 0.4) (the
    CPU restatement of this chain gives (1.187, 0.388), posterior sd 0.03); the same data read as right-censored at the
    last inspection passed put both rates below half of the truth."""
    import phasetype_b200 as pb
    a, c = 1.2, 0.4
    R = np.zeros((2, 2)); R[0, 1] = a; s = np.array([c, a])
    Tm = np.zeros((3, 3), dtype=np.int32); Tm[0, 1] = 1; Tm[1, 2] = 1; Tm[0, 2] = 2
    T = Tm.ravel(order="F").copy(); C = np.ones(9); truth = np.array([a, c])
    y, u, cens, _ = synth.inspection(R, s, 4000, 0.5, 8, np.random.default_rng(2024))
    means = {}
    for name, bounds in (("interval", u), ("right", None)):
        eng = pb.Engine(2, T, C, np.ones(2), np.ones(2), y, cens, method=1, mhit=1, seed=11, sum_y_global=_sum_max(y, u))
        if bounds is not None:
            eng.set_upper(bounds)
        eng.set_theta(np.ones(2), next_iter=1)
        means[name] = eng.run(399)[99:].mean(0)
        eng.close()
    assert (np.abs(means["interval"] / truth - 1.0) < 0.10).all(), means
    assert (means["right"] / truth < 0.5).all(), means


@pytest.mark.parametrize("method", [2, 4, 8, 16])
def test_other_methods_refuse_bounds(method):
    import phasetype_b200 as pb
    wl = synth.config(2, "ECS", l=200)
    eng = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, np.ones(wl.l, dtype=np.int32), method=method, seed=1)
    with pytest.raises(pb.EngineError, match="need method MHRS"):
        eng.set_upper(wl.y + 1.0)
    eng.close()


@pytest.mark.parametrize("case,msg", [("below", "not above y"), ("equal", "not above y"), ("exact", "exact observation"),
                                      ("nan", "NaN"), ("zbits", "too fine"), ("length", "bounds for")])
def test_bad_bounds_are_refused(case, msg):
    import phasetype_b200 as pb
    rng = np.random.default_rng(9)
    R, s = util.dense_rates(4, rng)
    T, C, theta = util.general_model(R, s)
    m = theta.shape[0]
    y = rng.exponential(1.0, 100) + 0.01
    cens = np.ones(100, dtype=np.int32); cens[:10] = 0
    u = np.full(100, np.inf); u[50:] = y[50:] + 1.0
    zbits = None
    if case == "below":
        u[60] = y[60] - 0.1
    elif case == "equal":
        u[60] = y[60]
    elif case == "exact":
        u[3] = y[3] + 1.0
    elif case == "nan":
        u[70] = np.nan
    elif case == "zbits":
        u[50:] = y[50:] + 1e6                              # paths end by u: far beyond what sum(y) leaves room for
    elif case == "length":
        u = u[:99]
    eng = pb.Engine(4, T, C, np.full(m, 2.0), np.full(m, 2.0), y, cens, method=1, seed=1, zbits=zbits)
    with pytest.raises(pb.EngineError, match=msg):
        eng.set_upper(u)
    eng.close()
