"""Groups of observations with their own structure over one parameter vector (pht_engine_set_groups), on the GPU: one group
is the plain engine bit for bit; every observation's path is the path a single-structure engine with its group's
structure draws; the per-group statistics are the sums of those paths; a grouped chain equals the host restatement
(oracle/pht_oracle_groups.c); chains x groups equal single-chain grouped engines; graph and direct launches agree; 64
chains recover a two-group posterior computed by quadrature; and the refusals."""
import numpy as np
import pytest

from phasetype_b200._lib import MAX_CHAINS, MAX_GROUPS, METHOD_UNIF
from phasetype_b200.diagnostics import split_rhat
from tests import util

pytestmark = pytest.mark.gpu

SWEEPS = 12


def _exit_groups(n, G, rng):
    """A dense n-phase structure whose transition rates are shared and whose exit rates differ by group: group 0 has n
    exit parameters, group g >= 1 exits at one parameter of its own times group 0's rates (held in C), so that m stays
    within the n(n+1) an engine takes.  Returns (T, C) of shape (G, (n+1)^2), column-major, and theta (the transition
    rates, group 0's exit rates, then the G - 1 exit scales)."""
    R, s = util.dense_rates(n, rng)
    T0, C0, theta0 = util.general_model(R, s)
    T0 = np.asarray(T0, dtype=np.int32).reshape(n + 1, n + 1, order="F")
    C0 = np.asarray(C0, dtype=np.float64).reshape(n + 1, n + 1, order="F")
    mt = int(theta0.shape[0]) - n                       # parameters are numbered column-major: the exits come last
    Ts, Cs = [], []
    for g in range(G):
        T, C = T0.copy(), C0.copy()
        if g:
            T[:n, n] = mt + n + g
            C[:n, n] = s
        Ts.append(T.ravel(order="F")); Cs.append(C.ravel(order="F"))
    theta = np.concatenate([theta0, rng.uniform(0.5, 2.0, G - 1)])
    return np.array(Ts), np.array(Cs), theta


def _mixed(l, rng):
    """A quarter each of exact, right-, interval- and left-censored observations."""
    y = rng.exponential(1.0, l) + 0.01
    kind = rng.integers(0, 4, l)
    cens = (kind > 0).astype(np.int32)
    y = np.where(kind == 3, 0.0, y)
    u = np.where(kind >= 2, y + rng.exponential(0.7, l) + 1e-3, np.inf)
    return y, cens, u


class Setup:
    def __init__(self, n, l, G, seed, chains=1, empty=()):
        rng = np.random.default_rng(seed)
        self.n, self.G = n, G
        self.T, self.C, self.theta = _exit_groups(n, G, rng)
        self.m = self.theta.shape[0]
        self.y, self.cens, self.u = _mixed(l, rng)
        live = [g for g in range(G) if g not in empty]
        self.group = np.array(live, dtype=np.int32)[rng.integers(0, len(live), l)]
        self.pi = rng.uniform(0.1, 1.0, n); self.pi /= self.pi.sum()
        self.beta = rng.uniform(0.5, 2.0, n)
        self.thetas = self.theta[None, :] * rng.uniform(0.5, 2.0, (chains, self.m))
        self.keys = np.array([0x9E3779B97F4A7C15 * (c + 3) % 2 ** 64 for c in range(chains)], dtype=np.uint64)
        self.sy = float(np.where(np.isfinite(self.u), self.u, self.y).sum())

    def engine(self, seed, T=None, C=None, upper=True, **kw):
        import phasetype_b200 as pb
        eng = pb.Engine(self.n, self.T[0] if T is None else T, self.C[0] if C is None else C, np.full(self.m, 2.0),
                        np.full(self.m, 2.0), self.y, self.cens, method=METHOD_UNIF, seed=int(seed), sum_y_global=self.sy, **kw)
        if upper:
            eng.set_upper(self.u)
        return eng

    def grouped(self, seed, **kw):
        eng = self.engine(seed, **kw)
        eng.set_groups(self.T, self.C, self.group)
        return eng


def test_one_group_is_the_plain_engine():
    st = Setup(4, 2000, 1, seed=1, chains=3)
    T, C = st.T[0], st.C[0]

    def run(eng, chains):
        if chains > 1:
            eng.set_chains(chains, st.keys)
            eng.set_chain_theta(st.thetas, next_iter=1)
        else:
            eng.set_theta(st.thetas[0], next_iter=1)
        eng.set_pi(st.pi, st.beta)
        th = eng.run_chains(SWEEPS)
        return th, eng.chain_pi_rows(SWEEPS)

    for chains in (1, 3):
        plain = st.engine(st.keys[0])
        want = run(plain, chains)
        plain.close()
        one = st.engine(st.keys[0])
        one.set_groups(T[None], C[None], np.zeros(2000, np.int32))
        got = run(one, chains)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
        one.set_groups(None)                         # back to the configured structure
        again = run(one, chains)
        assert np.array_equal(again[0], want[0]) and np.array_equal(again[1], want[1])
        one.close()


@pytest.mark.parametrize("n", [1, 4, 8, 32])
def test_paths_and_group_stats_are_each_groups_own(n):
    G = 2 if n == 1 else 3                           # m <= n(n+1)
    st = Setup(n, 1500 if n <= 8 else 500, G, seed=20 + n)
    eng = st.grouped(77)
    eng.set_theta(st.theta, next_iter=3)
    eng.set_pi(st.pi)
    B, N, z = eng.paths()
    Ng, Bg, zg = eng.group_stats()
    Ns, Bs, zs = eng.sweep_stats()
    zbits = eng.zbits
    eng.close()
    scale = 2.0 ** zbits
    for g in range(G):
        one = st.engine(77, T=st.T[g], C=st.C[g])
        one.set_theta(st.theta, next_iter=3)
        one.set_pi(st.pi)
        B1, N1, z1 = one.paths()
        one.close()
        k = st.group == g
        assert np.array_equal(B[k], B1[k]) and np.array_equal(N[k], N1[k]) and np.array_equal(z[k], z1[k]), "group %d" % g
        assert np.array_equal(Ng[g], N[k].sum(0).astype(np.int64))
        assert np.array_equal(Bg[g], np.bincount(B[k], minlength=n)[:n])
        assert np.array_equal(zg[g], np.rint(z[k] * scale).astype(np.int64).sum(0))
    assert np.array_equal(Ns, Ng.sum(0)) and np.array_equal(Bs, Bg.sum(0)) and np.array_equal(zs, zg.sum(0))


@pytest.mark.parametrize("G,empty", [(2, ()), (5, (3,))])
def test_chain_equals_host_restatement(G, empty):
    from oracle import pyoracle_groups as pg
    st = Setup(4, 800, G, seed=40 + G, empty=empty)
    eng = st.grouped(31)
    eng.set_theta(st.theta, next_iter=1)
    got = eng.run(20)
    zbits = eng.zbits
    eng.close()
    want = pg.gibbs_groups(31, 21, 4, np.full(st.m, 2.0), np.full(st.m, 2.0), st.T, st.C, st.y, st.cens, st.group, st.theta,
                           zbits, u=st.u)
    assert np.array_equal(got, want[1:])


@pytest.mark.parametrize("chains", [2, 64])
def test_chains_of_a_grouped_engine_equal_single_chain_grouped_engines(chains):
    st = Setup(4, 1500, 3, seed=60 + chains, chains=chains)
    eng = st.engine(1234)
    if chains == 2:                                  # both orders of the two calls
        eng.set_groups(st.T, st.C, st.group); eng.set_chains(chains, st.keys)
    else:
        eng.set_chains(chains, st.keys); eng.set_groups(st.T, st.C, st.group)
    eng.set_chain_theta(st.thetas, next_iter=1)
    eng.set_pi(st.pi, st.beta)
    th = eng.run_chains(SWEEPS)
    pi = eng.chain_pi_rows(SWEEPS)
    eng.close()
    for c in ((0, 1) if chains == 2 else (0, 1, 40, 63)):
        one = st.grouped(st.keys[c])
        one.set_theta(st.thetas[c], next_iter=1)
        one.set_pi(st.pi, st.beta)
        assert np.array_equal(one.run(SWEEPS), th[c]) and np.array_equal(one.pi_rows(SWEEPS), pi[c]), "chain %d" % c
        one.close()
    assert not np.array_equal(th[0], th[1])


def test_graph_and_direct_launches_agree():
    st = Setup(4, 2000, 4, seed=9, chains=5)
    out = []
    for graph in (True, False):
        eng = st.grouped(5, use_graph=graph)
        eng.set_chains(5, st.keys)
        eng.set_chain_theta(st.thetas, next_iter=1)
        eng.set_pi(st.pi, st.beta)
        out.append((eng.run_chains(SWEEPS), eng.chain_pi_rows(SWEEPS)))
        eng.close()
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])


def _quadrature_means(y0, exposure0, y1, c1, nu, zeta):
    """Posterior means of (theta1, theta2): group 0 exponential(theta1) with exact times y0 and total censored time
    exposure0, group 1 hypoexponential theta1 -> theta2 (exact y1[~c1], right-censored y1[c1]), Gamma(nu, zeta) priors;
    the log posterior on a grid, refined once around its mass."""
    def logpost(t1, t2):
        a1, a2 = t1[:, None], t2[None, :]
        d = a2 - a1
        lp = (nu - 1) * np.log(a1) - zeta * a1 + (nu - 1) * np.log(a2) - zeta * a2
        lp = lp + y0.size * np.log(a1) - a1 * (y0.sum() + exposure0)
        for v, cen in zip(y1, c1):
            e1 = np.exp(-a1 * v)
            a = e1 * np.where(d == 0.0, v, -np.expm1(-d * v) / np.where(d == 0.0, 1.0, d))   # (e^{-t1 v} - e^{-t2 v}) / (t2 - t1)
            lp = lp + np.log(e1 + a1 * a if cen else a1 * a2 * a)                            # S(v) or f(v)
        return lp
    t1, t2 = np.linspace(0.3, 3.0, 271), np.linspace(0.5, 12.0, 297)
    for _ in range(2):
        lp = logpost(t1, t2)
        w = np.exp(lp - lp.max()); w /= w.sum()
        m1, m2 = (w.sum(1) * t1).sum(), (w.sum(0) * t2).sum()
        s1 = np.sqrt((w.sum(1) * (t1 - m1) ** 2).sum()); s2 = np.sqrt((w.sum(0) * (t2 - m2) ** 2).sum())
        t1 = np.linspace(max(m1 - 8 * s1, 1e-3), m1 + 8 * s1, 301)
        t2 = np.linspace(max(m2 - 8 * s2, 1e-3), m2 + 8 * s2, 303)
    return m1, m2


def test_two_group_posterior_by_quadrature():
    """Group 0 exponential at theta1, group 1 two phases theta1 -> theta2: 64 chains against a 2-D quadrature."""
    import phasetype_b200 as pb
    from phasetype_b200 import synth
    rng = np.random.default_rng(77)
    n, nu, zeta = 2, 2.0, 1.0
    T = np.zeros((2, 3, 3), dtype=np.int32)
    T[0, 0, 2] = 1; T[0, 1, 2] = 1                    # group 0: exit at theta1 (phase 1 is never entered)
    T[1, 0, 1] = 1; T[1, 1, 2] = 2                    # group 1: theta1 to phase 1, exit at theta2
    T = np.array([t.ravel(order="F") for t in T]); C = np.ones((2, 9))
    y, cens, group = synth.groups(T, C, np.array([1.0, 2.5]), n, (300, 300), rng,
                                  censor=lambda k, r: r.uniform(0.5, 4.0, k))
    eng = pb.Engine(n, T[0], C[0], [nu, nu], [zeta, zeta], y, cens, method=METHOD_UNIF, seed=8, zbits=30)
    eng.set_groups(T, C, group)
    chains, sweeps = 64, 4000                         # the latent split of group 1's paths makes theta mix slowly
    eng.set_chains(chains)
    eng.set_chain_theta(np.exp(rng.uniform(np.log(0.3), np.log(6.0), (chains, 2))), next_iter=1)
    draws = eng.run_chains(sweeps)[:, sweeps // 2:, :]
    eng.close()
    k0, c = group == 0, cens.astype(bool)
    m1, m2 = _quadrature_means(y[k0 & ~c], float(y[k0 & c].sum()), y[~k0], c[~k0], nu, zeta)
    for p, want in ((0, m1), (1, m2)):
        cm = draws[:, :, p].mean(1)
        se = cm.std(ddof=1) / np.sqrt(chains)       # the 64 chains are independent
        assert abs(cm.mean() - want) < 5.0 * se + 1e-4 * want, (p, cm.mean(), want, se)
        assert split_rhat(draws[:, :, p]) < 1.01


def test_refusals():
    import phasetype_b200 as pb
    st = Setup(3, 600, 2, seed=3, chains=2)
    mh = pb.Engine(3, st.T[0], st.C[0], np.full(st.m, 2.0), np.full(st.m, 2.0), st.y[st.y > 0], st.cens[st.y > 0], method=1, seed=1)
    with pytest.raises(pb.EngineError, match="need method 64"):
        mh.set_groups(st.T, st.C, st.group[st.y > 0])
    mh.close()
    two = pb.Engine(3, st.T[0], st.C[0], np.full(st.m, 2.0), np.full(st.m, 2.0), st.y, st.cens, method=METHOD_UNIF, seed=1,
                    rank=0, world=2, sum_y_global=2 * st.sy)
    with pytest.raises(pb.EngineError, match="world = 1"):
        two.set_groups(st.T, st.C, st.group)
    two.close()
    eng = st.engine(1)
    eng.set_theta(st.theta, next_iter=1)
    want = eng.run(2)

    def same():
        eng.set_theta(st.theta, next_iter=1)
        assert np.array_equal(eng.run(2), want)

    for G in (0, MAX_GROUPS + 1):
        with pytest.raises(pb.EngineError, match="outside 1..%d" % MAX_GROUPS):
            eng.set_groups(np.tile(st.T[:1], (G, 1)), np.tile(st.C[:1], (G, 1)), np.zeros(600, np.int32))
    bad = st.T.copy(); bad[1, 0] = st.m + 1
    with pytest.raises(pb.EngineError, match="group 1: T\\[0\\] = %d outside 0..m" % (st.m + 1)):
        eng.set_groups(bad, st.C, st.group)
    bad = st.T.copy(); bad[0, 3] = 1                 # row n + 1 (the absorbing state), column 0
    with pytest.raises(pb.EngineError, match="absorbing state"):
        eng.set_groups(bad, st.C, st.group)
    with pytest.raises(pb.EngineError, match="is used by no group"):
        eng.set_groups(st.T[:1], st.C[:1], np.zeros(600, np.int32))    # group 1's exit parameters unused
    g = st.group.copy(); g[17] = 2
    with pytest.raises(pb.EngineError, match="group\\[17\\] = 2 outside 0..1"):
        eng.set_groups(st.T, st.C, g)
    same()
    # chains x groups
    eng.set_chains(MAX_CHAINS // 32 + 1)
    with pytest.raises(pb.EngineError, match="exceeds %d" % MAX_CHAINS):
        eng.set_groups(np.tile(st.T, (16, 1)), np.tile(st.C, (16, 1)), st.group)
    eng.set_chains(1)
    eng.set_groups(st.T, st.C, st.group)
    with pytest.raises(pb.EngineError, match="chains x groups = %d x 2 exceeds" % MAX_CHAINS):
        eng.set_chains(MAX_CHAINS)
    # entry ages, in either order
    a = np.where(st.y > 0, st.y / 4, 0.0)
    eng.set_upper(None)
    with pytest.raises(pb.EngineError, match="not supported with 2 groups"):
        eng.set_entry(a)
    eng.set_groups(None)
    eng.set_entry(a)
    with pytest.raises(pb.EngineError, match="entry ages"):
        eng.set_groups(st.T, st.C, st.group)
    eng.set_entry(None)
    eng.set_upper(st.u)
    same()
    eng.close()


def test_failed_allocation_is_refused_and_leaves_the_engine_as_it_was():
    """16 chains x 64 groups at n = 32 need about 34 GB of tables; with less than that free the call fails."""
    import torch

    import phasetype_b200 as pb
    st = Setup(32, 300, 1, seed=32, chains=16)
    eng = st.engine(11)
    eng.set_theta(st.theta, next_iter=1)
    want = eng.run(2)
    eng.set_chains(16)
    pb.lib().pht_release_device_memory()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    hold = torch.empty(max(free - (16 << 30), 0), dtype=torch.uint8, device="cuda")       # leave 16 GB free
    try:
        with pytest.raises(pb.EngineError, match="cannot allocate device memory for 64 groups"):
            eng.set_groups(np.tile(st.T, (64, 1)), np.tile(st.C, (64, 1)), np.zeros(300, np.int32))
    finally:
        del hold
        torch.cuda.empty_cache()
    assert eng.groups == 1
    eng.set_chains(1)
    eng.set_theta(st.theta, next_iter=1)
    assert np.array_equal(eng.run(2), want)
    eng.close()
