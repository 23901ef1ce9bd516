"""The uniformisation path sampler on the device (method 64, k_unif.cu): per-observation parity with the host build of
the sampler (oracle/pht_oracle_unif.c) for every kind of observation, sweep statistics and chains, several GPUs,
LJMA_Gibbs, tier 2 on generators the spectral samplers cannot carry, recovery of rates and of pi, and the refusals."""
import os
import threading

import numpy as np
import pytest

from oracle import pyoracle as po
from oracle import pyoracle_unif as pu
from phasetype_b200 import synth
from phasetype_b200._lib import METHOD_UNIF
from tests import util

pytestmark = pytest.mark.gpu


def _mixed(n, l, rng):
    """Dense n-phase model; a quarter each of exact, right-, interval- and left-censored observations."""
    R, s = util.dense_rates(n, rng)
    y = rng.exponential(1.0, l) + 0.01
    kind = rng.integers(0, 4, l)
    cens = (kind > 0).astype(np.int32)
    y = np.where(kind == 3, 0.0, y)
    u = np.where(kind >= 2, y + rng.exponential(0.7, l) + 1e-3, np.inf)
    return R, s, y, cens, u


def _sum_max(y, u):
    return float(np.where(np.isfinite(u), u, y).sum())


def _engine(R, s, y, cens, u=None, seed=7, **kw):
    import phasetype_b200 as pb
    n = s.shape[0]
    T, C, theta = util.general_model(R, s)
    m = theta.shape[0]
    eng = pb.Engine(n, T, C, np.full(m, 2.0), np.full(m, 2.0), y, cens, method=METHOD_UNIF, seed=seed,
                    sum_y_global=_sum_max(y, u) if u is not None else float(y.sum()), **kw)
    if u is not None:
        eng.set_upper(u)
    return eng, T, C, theta


@pytest.mark.parametrize("n,l,general_pi", [(1, 200000, False), (3, 200000, True), (4, 200000, False), (8, 200000, True),
                                            (16, 20000, False), (16, 20000, True), (32, 8000, False), (32, 8000, True)])
def test_paths_match_oracle(n, l, general_pi):
    """Exact, right-, interval- and left-censored observations; shards with more observations than resident lanes
    (n <= 8), so that warps take a second chunk."""
    rng = np.random.default_rng(100 + n)
    R, s, y, cens, u = _mixed(n, l, rng)
    eng, _, _, theta = _engine(R, s, y, cens, u, seed=0xC0FFEE)
    pi = None
    if general_pi:
        pi = rng.uniform(0.1, 1.0, n); pi /= pi.sum()
        eng.set_pi(pi)
    eng.set_theta(theta, next_iter=4)
    B, N, z = eng.paths()
    mdl = eng.model()
    eng.close()
    Bo, No, zo, err = pu.unif_paths(0xC0FFEE, 4, y, cens, mdl["S"], mdl["s"], u=u, pi=pi)
    assert err == 0
    assert np.array_equal(B, Bo)
    assert np.array_equal(N, No)
    assert np.array_equal(z, zo)


def test_sweep_stats_c3_match_oracle():
    """10^6 observations of the C3 shape (20 % right-censored) in the production layout (decreasing y)."""
    import phasetype_b200 as pb
    wl = synth.config(3, "MHRS", l=10 ** 6)
    eng = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=METHOD_UNIF, seed=2718)
    eng.set_theta(wl.theta, next_iter=3)
    N, B, z = eng.sweep_stats()
    zbits = eng.zbits
    eng.close()
    No, Bo, zo = pu.unif_sweep_stats(2718, 3, True, wl.n, wl.T, wl.C, wl.theta, wl.y, wl.censored, zbits)
    assert np.array_equal(N, No) and np.array_equal(B, Bo) and np.array_equal(z, zo)


def _chain_workload(l=20000):
    rng = np.random.default_rng(12)
    R, s, y, cens, u = _mixed(5, l, rng)
    T, C, theta = util.general_model(R, s)
    return R, s, y, cens, u, T, C, theta


def test_chain_equals_oracle():
    import phasetype_b200 as pb
    R, s, y, cens, u, T, C, theta = _chain_workload()
    m = theta.shape[0]
    eng = pb.Engine(5, T, C, np.full(m, 2.0), np.full(m, 2.0), y, cens, method=METHOD_UNIF, seed=31, sum_y_global=_sum_max(y, u))
    eng.set_upper(u)
    eng.set_theta(theta, next_iter=1)
    got = eng.run(20)
    zbits = eng.zbits
    eng.close()
    want = pu.gibbs_unif(31, 21, 5, np.full(m, 2.0), np.full(m, 2.0), T, C, y, cens, theta, zbits, u=u)
    assert np.array_equal(got, want[1:])


def test_two_gpus_equal_one():
    import phasetype_b200 as pb
    if pb.lib().pht_device_count() < 2:
        pytest.skip("needs two or more GPUs")
    R, s, y, cens, u, T, C, theta = _chain_workload(40000)
    m = theta.shape[0]
    sy = _sum_max(y, u)

    def engine(rank, world):
        e = pb.Engine(5, T, C, np.full(m, 2.0), np.full(m, 2.0), y[rank::world], cens[rank::world], method=METHOD_UNIF, seed=8,
                      device=rank, rank=rank, world=world, use_graph=False, sum_y_global=sy)
        e.set_upper(u[rank::world])
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


def test_ljma_gibbs_equals_engine_chain():
    import phasetype_b200 as pb
    wl = synth.config(3, "MHRS", l=5000)
    os.environ["PHT_B200_SEED"] = "777"; os.environ["PHT_B200_QUIET"] = "1"; os.environ["PHT_B200_GRAPH"] = "1"
    res = pb.ljma_gibbs(8, 1, METHOD_UNIF, wl.n, wl.m, wl.nu, wl.zeta, wl.T, wl.C, wl.y, wl.censored, [-1.0])
    start = (wl.nu - 1.0) / wl.zeta
    eng = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=METHOD_UNIF, seed=777)
    eng.set_theta(start, next_iter=1)
    got = eng.run(7)
    zbits = eng.zbits
    eng.close()
    assert np.array_equal(res[0], start) and np.array_equal(res[1:], got)
    want = pu.gibbs_unif(777, 8, wl.n, wl.nu, wl.zeta, wl.T, wl.C, wl.y, wl.censored, start, zbits)
    assert np.array_equal(res, want)


ERLANG4 = (np.diag(np.full(3, 2.0), 1), np.array([0.0, 0.0, 0.0, 2.0]))
TIED_COXIAN = (np.diag(np.full(3, 1.5), 1), np.array([0.3, 0.3, 0.3, 1.5]))


@pytest.mark.parametrize("name", ["erlang4", "tied_coxian"])
def test_tier2_where_spectral_samplers_fail(name):
    """Exact observations at y = 2 of generators with a Jordan block: the mean sojourns match the Van Loan integrals."""
    from tests.test_unif_oracle import expectations
    R, s = ERLANG4 if name == "erlang4" else TIED_COXIAN
    l = 200000
    y = np.full(l, 2.0); cens = np.zeros(l, dtype=np.int32)
    eng, _, _, theta = _engine(R, s, y, cens, seed=3)
    eng.set_theta(theta, next_iter=1)
    B, N, z = eng.paths()
    mdl = eng.model()
    eng.close()
    Sm = mdl["S"].reshape(4, 4, order="F")
    Ez, EN, Eexit, _ = expectations(Sm, mdl["s"], np.eye(4)[0], 2.0, "exact")
    assert (np.abs(z.mean(0) - Ez) < 4.5 * z.std(0) / np.sqrt(l) + 2e-4).all(), (z.mean(0), Ez)
    Nm = N.reshape(l, 4, 4).transpose(0, 2, 1)
    ex = np.diagonal(Nm, axis1=1, axis2=2)
    assert (np.abs(ex.mean(0) - Eexit) < 4.5 * ex.std(0) / np.sqrt(l) + 2e-4).all()
    if name == "erlang4":
        assert np.allclose(z.mean(0), 0.5, atol=0.01)


def _tied_model():
    """Tied Coxian (the generator of TIED_COXIAN): phases 1-3 move on at F and exit at R, phase 4 exits at F
    (parameters 1 = F, 2 = R).  (With the exit rate R from every phase the absorption time would be Exp(R) whatever F.)"""
    n = 4
    Tm = np.zeros((n + 1, n + 1), dtype=np.int32)
    for i in range(n - 1):
        Tm[i, i + 1] = 1; Tm[i, n] = 2
    Tm[n - 1, n] = 1
    return Tm.ravel(order="F").copy(), np.ones((n + 1) ** 2)


def test_rates_recovered_from_tied_coxian_data():
    import phasetype_b200 as pb
    F, Rx = 1.5, 0.3
    Rm = np.diag(np.full(3, F), 1); s = np.array([Rx, Rx, Rx, F])
    y = synth.simulate_pht(Rm, s, 20000, np.random.default_rng(77))
    T, C = _tied_model()
    eng = pb.Engine(4, T, C, np.ones(2), np.ones(2), y, np.zeros(y.shape[0], dtype=np.int32), method=METHOD_UNIF, seed=5)
    eng.set_theta(np.ones(2), next_iter=1)
    mean = eng.run(300)[100:].mean(0)
    eng.close()
    assert (np.abs(mean / np.array([F, Rx]) - 1.0) < 0.1).all(), mean


def test_rates_recovered_from_inspection_data_with_left_censoring():
    """Inspection data whose first interval is (0, spacing]: left-censored, y = 0."""
    import phasetype_b200 as pb
    a, c = 1.2, 0.4
    R = np.zeros((2, 2)); R[0, 1] = a; s = np.array([c, a])
    Tm = np.zeros((3, 3), dtype=np.int32); Tm[0, 1] = 1; Tm[1, 2] = 1; Tm[0, 2] = 2
    T = Tm.ravel(order="F").copy(); C = np.ones(9); truth = np.array([a, c])
    y, u, cens, _ = synth.inspection(R, s, 4000, 0.5, 8, np.random.default_rng(2024))
    y = np.where(y < 1e-6, 0.0, y)
    assert (y == 0).sum() > 100
    eng = pb.Engine(2, T, C, np.ones(2), np.ones(2), y, cens, method=METHOD_UNIF, seed=11, sum_y_global=_sum_max(y, u))
    eng.set_upper(u)
    eng.set_theta(np.ones(2), next_iter=1)
    mean = eng.run(400)[100:].mean(0)
    eng.close()
    assert (np.abs(mean / truth - 1.0) < 0.10).all(), mean


def test_dirichlet_update_recovers_pi():
    """Two parallel exponential phases (exit rates 0.5 and 3) entered with pi = (0.3, 0.7)."""
    import phasetype_b200 as pb
    rng = np.random.default_rng(8)
    l = 20000
    start = rng.uniform(size=l) < 0.7
    y = rng.exponential(1.0, l) / np.where(start, 3.0, 0.5)
    Tm = np.zeros((3, 3), dtype=np.int32); Tm[0, 2] = 1; Tm[1, 2] = 2
    eng = pb.Engine(2, Tm.ravel(order="F").copy(), np.ones(9), np.ones(2), np.ones(2), y, np.zeros(l, dtype=np.int32),
                    method=METHOD_UNIF, seed=9)
    eng.set_pi(np.array([0.5, 0.5]), beta=np.ones(2))
    eng.set_theta(np.array([0.4, 2.5]), next_iter=1)      # (started on the labelling of the truth)
    th = eng.run(400)
    pis = eng.pi_rows(400)
    eng.close()
    assert np.allclose(pis[100:].mean(0), [0.3, 0.7], atol=0.04), pis[100:].mean(0)
    assert np.allclose(th[100:].mean(0), [0.5, 3.0], rtol=0.1), th[100:].mean(0)


def test_table_overflow_raises_bit_256():
    import phasetype_b200 as pb
    R = np.array([[0.0, 40.0], [0.0, 0.0]]); s = np.array([0.0, 1.0])
    y = np.array([1.0, 200.0]); cens = np.zeros(2, dtype=np.int32)
    eng, _, _, theta = _engine(R, s, y, cens)
    eng.set_theta(theta, next_iter=1)
    with pytest.raises(pb.EngineError, match="0x100.*more powers of R than its table holds"):
        eng.run(1)
    eng.close()


@pytest.mark.parametrize("case,msg", [("below", "not above y"), ("equal", "not above y"), ("exact", "exact observation"),
                                      ("nan", "NaN"), ("negative", "y >= 0")])
def test_bad_bounds_are_refused(case, msg):
    import phasetype_b200 as pb
    rng = np.random.default_rng(9)
    R, s = util.dense_rates(3, rng)
    y = rng.exponential(1.0, 50) + 0.01
    cens = np.ones(50, dtype=np.int32); cens[:5] = 0
    u = np.full(50, np.inf); u[20:] = y[20:] + 1.0
    if case == "below":
        u[30] = y[30] - 0.1
    elif case == "equal":
        u[30] = y[30]
    elif case == "exact":
        u[2] = y[2] + 1.0
    elif case == "nan":
        u[40] = np.nan
    elif case == "negative":
        y[30] = -0.5
    eng, _, _, _ = _engine(R, s, y, cens)
    with pytest.raises(pb.EngineError, match=msg):
        eng.set_upper(u)
    eng.close()


def test_spectral_override_refused():
    import phasetype_b200 as pb
    R, s = util.dense_rates(3, np.random.default_rng(1))
    eng, _, _, _ = _engine(R, s, np.ones(4), np.zeros(4, dtype=np.int32))
    with pytest.raises(pb.EngineError, match="no spectral data"):
        eng.set_spectral(np.ones(3), np.eye(3), np.eye(3))
    eng.close()
