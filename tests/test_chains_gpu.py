"""Several chains in one method-64 engine (pht_engine_set_chains): every chain equals, bit for bit, the chain of a
single-chain engine built with its key, for every kind of observation, a general pi with its Dirichlet update, more chains
than resident blocks and small shards; graph and direct launches agree; set_chains(1) is the single-chain engine; 64
chains recover the closed-form posterior of the exponential model and mix (split-R-hat); and the refusals."""
import numpy as np
import pytest

from phasetype_b200._lib import MAX_CHAINS, METHOD_UNIF
from phasetype_b200.diagnostics import split_rhat
from tests import util

pytestmark = pytest.mark.gpu

SWEEPS = 12


def _mixed(n, l, rng):
    """Dense n-phase model; a quarter each of exact, right-, interval- and left-censored observations."""
    R, s = util.dense_rates(n, rng)
    y = rng.exponential(1.0, l) + 0.01
    kind = rng.integers(0, 4, l)
    cens = (kind > 0).astype(np.int32)
    y = np.where(kind == 3, 0.0, y)
    u = np.where(kind >= 2, y + rng.exponential(0.7, l) + 1e-3, np.inf)
    return R, s, y, cens, u


class Setup:
    """One data set, model, pi prior and a theta per chain."""

    def __init__(self, n, l, chains, seed):
        rng = np.random.default_rng(seed)
        self.n = n
        R, s, self.y, self.cens, self.u = _mixed(n, l, rng)
        self.T, self.C, theta = util.general_model(R, s)
        self.m = theta.shape[0]
        self.thetas = theta[None, :] * rng.uniform(0.5, 2.0, (chains, self.m))
        self.pi = rng.uniform(0.1, 1.0, n); self.pi /= self.pi.sum()
        self.beta = rng.uniform(0.5, 2.0, n)
        self.keys = np.array([0x9E3779B97F4A7C15 * (c + 1) % 2 ** 64 for c in range(chains)], dtype=np.uint64)

    def engine(self, seed, **kw):
        import phasetype_b200 as pb
        sy = float(np.where(np.isfinite(self.u), self.u, self.y).sum())
        eng = pb.Engine(self.n, self.T, self.C, np.full(self.m, 2.0), np.full(self.m, 2.0), self.y, self.cens,
                        method=METHOD_UNIF, seed=int(seed), sum_y_global=sy, **kw)
        eng.set_upper(self.u)
        eng.set_pi(self.pi, self.beta)
        return eng

    def single(self, c, **kw):
        """SWEEPS sweeps of chain c by a single-chain engine with key keys[c]: (theta rows, pi rows)."""
        eng = self.engine(self.keys[c], **kw)
        eng.set_theta(self.thetas[c], next_iter=1)
        th = eng.run(SWEEPS)
        pi = eng.pi_rows(SWEEPS)
        eng.close()
        return th, pi

    def multi(self, **kw):
        eng = self.engine(1234, **kw)
        eng.set_chains(len(self.keys), self.keys)
        eng.set_chain_theta(self.thetas, next_iter=1)
        th = eng.run_chains(SWEEPS)
        pi = eng.chain_pi_rows(SWEEPS)
        eng.close()
        return th, pi


def _check_against_single(st, th, pi, which):
    for c in which:
        th1, pi1 = st.single(c)
        assert np.array_equal(th[c], th1), "chain %d: theta differs from its single-chain engine" % c
        assert np.array_equal(pi[c], pi1), "chain %d: pi differs from its single-chain engine" % c


@pytest.mark.parametrize("n", [1, 4, 8, 32])
@pytest.mark.parametrize("chains", [2, 5, 64])
def test_chains_equal_single_chain_engines(n, chains):
    st = Setup(n, 3000 if n <= 8 else 800, chains, seed=40 + n + chains)
    th, pi = st.multi()
    assert th.shape == (chains, SWEEPS, st.m) and pi.shape == (chains, SWEEPS, n)
    _check_against_single(st, th, pi, range(chains) if chains <= 5 else (0, 1, 31, 63))
    assert not np.array_equal(th[0], th[1])


def test_more_chains_than_resident_blocks():
    st = Setup(2, 3000, 600, seed=600)
    th, pi = st.multi()
    _check_against_single(st, th, pi, (0, 1, 599))


@pytest.mark.parametrize("l", [1, 31, 33, 1000])
def test_small_shards(l):
    st = Setup(4, l, 7, seed=70 + l)
    th, pi = st.multi()
    _check_against_single(st, th, pi, (0, 3, 6))


def test_graph_and_direct_launches_agree():
    st = Setup(4, 2000, 9, seed=9)
    th_g, pi_g = st.multi()
    th_d, pi_d = st.multi(use_graph=False)
    assert np.array_equal(th_g, th_d) and np.array_equal(pi_g, pi_d)


def test_one_chain_again_is_the_single_chain_engine():
    st = Setup(4, 2000, 6, seed=16)
    plain = st.engine(77)
    plain.set_theta(st.thetas[0], next_iter=1)
    want, want_pi = plain.run(SWEEPS), plain.pi_rows(SWEEPS)
    plain.close()
    eng = st.engine(77)
    eng.set_chains(6)
    eng.set_chain_theta(st.thetas, next_iter=1)
    many = eng.run_chains(SWEEPS)
    assert np.array_equal(many[0], want) and np.array_equal(eng.run(0), np.zeros((0, st.m)))
    eng.set_chains(1)
    eng.set_pi(st.pi, st.beta)
    eng.set_theta(st.thetas[0], next_iter=1)
    got = eng.run(SWEEPS)
    assert np.array_equal(got, want) and np.array_equal(eng.pi_rows(SWEEPS), want_pi)
    assert np.array_equal(eng.run_chains(0), np.zeros((1, 0, st.m)))
    eng.close()


def test_chain_zero_is_what_the_single_chain_calls_see():
    st = Setup(4, 2000, 5, seed=55)
    eng = st.engine(1234)
    eng.set_chains(5, st.keys)
    eng.set_chain_theta(st.thetas, next_iter=1)
    out = eng.run(SWEEPS)                           # run's out: chain 0
    th = np.zeros((5, SWEEPS, st.m))
    from phasetype_b200 import _lib
    _lib._check(_lib.lib().pht_engine_chain_rows(eng._h, SWEEPS, th.ctypes.data, None))
    assert np.array_equal(out, th[0])
    assert np.array_equal(eng.get_theta(), th[0, -1]) and np.array_equal(eng.get_chain_theta(), th[:, -1])
    assert np.array_equal(eng.pi_rows(SWEEPS), eng.chain_pi_rows(SWEEPS)[0])
    # set_theta sets every chain; the parity hooks draw chain 0 only and leave its stats identical to one chain's
    eng.set_theta(st.thetas[2], next_iter=3)
    eng.set_pi(st.pi, st.beta)                      # the run drew new pi; start the hooks from the fresh engine's
    assert np.array_equal(eng.get_chain_theta(), np.repeat(st.thetas[2][None, :], 5, axis=0))
    N, B, z = eng.sweep_stats()
    Bp, Np, zp = eng.paths()
    eng.close()
    one = st.engine(st.keys[0])
    one.set_theta(st.thetas[2], next_iter=3)
    N1, B1, z1 = one.sweep_stats()
    Bp1, Np1, zp1 = one.paths()
    one.close()
    assert np.array_equal(N, N1) and np.array_equal(B, B1) and np.array_equal(z, z1)
    assert np.array_equal(Bp, Bp1) and np.array_equal(Np, Np1) and np.array_equal(zp, zp1)


def test_exponential_posterior_from_overdispersed_starts():
    """n = 1: theta | y ~ Gamma(nu + d, zeta + sum y) with d exact observations (right-censored ones add their y)."""
    import phasetype_b200 as pb
    rng = np.random.default_rng(2024)
    l, rate, nu, zeta = 1000, 1.7, 2.0, 1.0
    t = rng.exponential(1.0 / rate, l)
    c = rng.uniform(0.0, 2.0, l)
    y = np.minimum(t, c); cens = (t > c).astype(np.int32)
    T = np.array([0, 0, 1, 0], dtype=np.int32); Cm = np.ones(4)
    # zbits 30: a chain started at theta = 0.01 draws censored sojourns of mean 100 in its first sweeps
    eng = pb.Engine(1, T, Cm, [nu], [zeta], y, cens, method=METHOD_UNIF, seed=5, zbits=30)
    chains, sweeps = 64, 2000
    eng.set_chains(chains)
    eng.set_chain_theta(np.geomspace(0.01, 100.0, chains)[:, None], next_iter=1)
    draws = eng.run_chains(sweeps)
    eng.close()
    shape, post_rate = nu + float(l - cens.sum()), zeta + float(y.sum())
    mean, var = shape / post_rate, shape / post_rate ** 2
    kept = draws[:, sweeps // 2:, 0]
    pooled = kept.ravel()
    se = np.sqrt(var / (pooled.size / 4.0))        # a quarter of the draws as effective: the censored sojourns correlate sweeps
    assert abs(pooled.mean() - mean) < 5.0 * se
    assert abs(pooled.var() / var - 1.0) < 0.05
    assert split_rhat(kept) < 1.01


def test_refusals():
    import phasetype_b200 as pb
    st = Setup(3, 500, 2, seed=3)
    sy = float(np.where(np.isfinite(st.u), st.u, st.y).sum())
    mh = pb.Engine(3, st.T, st.C, np.full(st.m, 2.0), np.full(st.m, 2.0), st.y[st.u == np.inf], st.cens[st.u == np.inf],
                   method=1, seed=1)
    with pytest.raises(pb.EngineError, match="need method 64"):
        mh.set_chains(2)
    mh.close()
    two = pb.Engine(3, st.T, st.C, np.full(st.m, 2.0), np.full(st.m, 2.0), st.y, st.cens, method=METHOD_UNIF, seed=1,
                    rank=0, world=2, sum_y_global=2 * sy)
    with pytest.raises(pb.EngineError, match="world = 1"):
        two.set_chains(2)
    two.close()
    eng = st.engine(1)
    for bad in (0, -1, MAX_CHAINS + 1):
        with pytest.raises(pb.EngineError, match="outside 1..%d" % MAX_CHAINS):
            eng.set_chains(bad)
    with pytest.raises(pb.EngineError, match="duplicate key"):
        eng.set_chains(3, [5, 6, 5])
    # delayed entry, in either order
    a = np.where(st.y > 0, st.y / 4, 0.0)
    eng.set_upper(None)
    eng.set_entry(a)
    with pytest.raises(pb.EngineError, match="entry ages"):
        eng.set_chains(2)
    eng.set_chains(1)                                # one chain keeps the entry ages
    eng.set_entry(None)
    eng.set_chains(2)
    with pytest.raises(pb.EngineError, match="not supported with 2 chains"):
        eng.set_entry(a)
    eng.set_chains(1)
    eng.set_entry(a)
    eng.set_theta(st.thetas[0], next_iter=1)
    assert np.isfinite(eng.run(2)).all()
    eng.close()


def test_failed_allocation_is_refused_and_leaves_the_engine_as_it_was():
    """1024 chains at n = 32 need about 37 GB of tables; with less than that free the call fails and one chain still runs."""
    import torch

    import phasetype_b200 as pb
    st = Setup(32, 200, 1, seed=32)
    eng = st.engine(11)
    eng.set_theta(st.thetas[0], next_iter=1)
    want = eng.run(2)
    eng.set_theta(st.thetas[0], next_iter=1)
    eng.set_pi(st.pi, st.beta)                      # the run drew new pi
    pb.lib().pht_release_device_memory()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    hold = torch.empty(max(free - (16 << 30), 0), dtype=torch.uint8, device="cuda")       # leave 16 GB free
    try:
        with pytest.raises(pb.EngineError, match="cannot allocate device memory for 1024 chains"):
            eng.set_chains(MAX_CHAINS)
    finally:
        del hold
        torch.cuda.empty_cache()
    assert eng.chains == 1
    assert np.array_equal(eng.run(2), want)
    eng.close()
