"""Misclassified panel observations (pht_engine_set_stage_visits) on the GPU: every path, the sweep statistics and the
emission counts K equal the host build (oracle/pht_oracle_misclass.c) bit for bit; a chain with a prior on E equals the host
chain (theta, pi and E rows); chain c equals the single-chain engine with key c; an indicator E equals the stage masks bit
for bit, alone and with chains, groups, delayed entry and interval bounds; observations without visits draw their old
paths; a progressive Coxian read with misreadings is recovered; and the refusals, each leaving the engine as it was."""
import numpy as np
import pytest

from oracle import pyoracle_misclass as pm
from phasetype_b200 import synth
from phasetype_b200._lib import MAX_STAGES, MAX_VISITS, METHOD_UNIF, EngineError
from tests import util

pytestmark = pytest.mark.gpu


def _data(n, S, l, rng, frac=0.6):
    """Exact, right-, interval- and left-censored observations; a share frac of them (y > 0) with 1..5 visits at sorted
    times in [0, y] (some at 0 and at y), each reading a random stage in 0..S-1."""
    y = rng.exponential(1.0, l) + 0.01
    kind = rng.integers(0, 4, l)
    cens = (kind > 0).astype(np.int32)
    y = np.where(kind == 3, 0.0, y)
    u = np.where(kind >= 2, y + rng.exponential(0.7, l) + 1e-3, np.inf)
    offs, ts = [0], []
    for k in range(l):
        m = 0
        if y[k] == 0.0:
            if rng.random() < 0.3:
                ts.append(0.0); m = 1
        elif rng.random() < frac:
            m = int(rng.integers(1, 6))
            t = np.sort(rng.uniform(0.0, y[k], m))
            if rng.random() < 0.2:
                t[0] = 0.0
            if rng.random() < 0.2:
                t[-1] = y[k]
            t = np.unique(t); m = t.shape[0]
            ts.extend(t.tolist())
        offs.append(offs[-1] + m)
    off = np.array(offs, dtype=np.int64)
    return y, cens, u, off, np.array(ts), rng.integers(0, S, int(off[-1])).astype(np.uint32)


def _emission(n, S, rng):
    """A dense E with a few structural zeros; every column keeps a positive entry."""
    E = rng.dirichlet(np.ones(S), n)
    if S > 1:
        for c in range(0, n, 3):
            o = (c // 3) % S
            if E[:, o].astype(bool).sum() > 1:
                E[c, o] = 0.0
        E /= E.sum(1, keepdims=True)
    return E


class Setup:
    def __init__(self, n, S, l, seed):
        rng = np.random.default_rng(seed)
        self.n, self.S = n, S
        R, s = util.dense_rates(n, rng)
        self.T, self.C, self.theta = util.general_model(R, s)
        self.m = self.theta.shape[0]
        self.y, self.cens, self.u, self.off, self.t, self.stage = _data(n, S, l, rng)
        self.E = _emission(n, S, rng)
        self.alpha = np.where(self.E > 0, rng.uniform(0.5, 3.0, self.E.shape), 0.0)
        self.pi = rng.uniform(0.1, 1.0, n); self.pi /= self.pi.sum()
        self.beta = rng.uniform(0.5, 2.0, n)
        self.sy = float(np.where(np.isfinite(self.u), self.u, self.y).sum())

    def engine(self, seed, visits=True, alpha=False, **kw):
        import phasetype_b200 as pb
        eng = pb.Engine(self.n, self.T, self.C, np.full(self.m, 2.0), np.full(self.m, 2.0), self.y, self.cens,
                        method=METHOD_UNIF, seed=int(seed), sum_y_global=self.sy, **kw)
        eng.set_upper(self.u)
        eng.set_pi(self.pi)
        if visits:
            eng.set_stage_visits(self.E, self.off, self.t, self.stage, alpha=self.alpha if alpha else None)
        return eng


@pytest.mark.parametrize("n,S", [(1, 1), (4, 3), (8, 2), (8, 8), (32, 5)])
def test_paths_stats_and_counts_equal_the_host_build(n, S):
    st = Setup(n, S, 1200 if n <= 8 else 300, seed=60 + n + S)
    eng = st.engine(93)
    eng.set_theta(st.theta, next_iter=5)
    got = eng.paths()
    mdl = eng.model()
    *want, err = pm.misclass_paths(93, 5, st.y, st.cens, st.off, st.t, st.stage, st.E, mdl["S"], mdl["s"], u=st.u, pi=st.pi)
    assert err == 0
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
    eng.set_theta(st.theta, next_iter=6)
    N, B, z = eng.sweep_stats()
    eng.set_theta(st.theta, next_iter=6)
    K = eng.emission_stats()
    zbits = eng.zbits
    eng.close()
    No, Bo, zo, Ko = pm.misclass_sweep_stats(93, 6, True, n, st.T, st.C, st.theta, st.y, st.cens, st.off, st.t, st.stage,
                                             st.E, zbits, u=st.u, pi=st.pi)
    assert np.array_equal(N, No) and np.array_equal(B, Bo) and np.array_equal(z, zo) and np.array_equal(K, Ko)
    assert K.sum() == st.off[-1]


@pytest.mark.parametrize("graph", [True, False])
def test_chain_with_prior_equals_host_chain(graph):
    st = Setup(4, 3, 1500, seed=7)
    start = st.theta * 1.3
    eng = st.engine(31, alpha=True, use_graph=graph)
    eng.set_theta(start, next_iter=1)
    eng.set_pi(st.pi, st.beta)
    got = eng.run(20)
    pis, Es = eng.pi_rows(20), eng.emission_rows(20)[0]
    last = eng.emission()
    zbits = eng.zbits
    eng.close()
    want, wpi, wE = pm.gibbs_misclass(31, 21, st.n, np.full(st.m, 2.0), np.full(st.m, 2.0), st.T, st.C, st.y, st.cens, st.off,
                                      st.t, st.stage, st.E, start, zbits, u=st.u, pi=st.pi, beta=st.beta, alpha=st.alpha)
    assert np.array_equal(got, want[1:]) and np.array_equal(pis, wpi[1:]) and np.array_equal(Es, wE[1:])
    assert np.array_equal(last, wE[-1]) and not np.array_equal(last, st.E)
    assert ((Es > 0) == (st.alpha > 0)[None]).all()


@pytest.mark.parametrize("order", ["visits_first", "chains_first"])
def test_chains_equal_single_chain_engines(order):
    st = Setup(4, 3, 1500, seed=9)
    keys = np.array([11, 2 ** 40 + 3, 77], dtype=np.uint64)
    thetas = st.theta[None, :] * np.array([[0.8], [1.0], [1.3]])
    eng = st.engine(keys[0], visits=order == "visits_first", alpha=True)
    eng.set_chains(3, keys)
    if order == "chains_first":
        eng.set_stage_visits(st.E, st.off, st.t, st.stage, alpha=st.alpha)
    eng.set_chain_theta(thetas, next_iter=1)
    eng.set_pi(st.pi, st.beta)
    got = eng.run_chains(6), eng.chain_pi_rows(6), eng.emission_rows(6)
    eng.close()
    for c in range(3):
        one = st.engine(keys[c], alpha=True)
        one.set_theta(thetas[c], next_iter=1)
        one.set_pi(st.pi, st.beta)
        assert np.array_equal(got[0][c], one.run(6)) and np.array_equal(got[1][c], one.pi_rows(6))
        assert np.array_equal(got[2][c], one.emission_rows(6)[0])
        one.close()


def test_groups_and_chains_with_prior_equal_the_host_chain():
    """Two groups with their own structure and two chains, E drawn: K is summed over the groups into one block per chain,
    and chain c equals the grouped host chain with key c (theta, pi and E rows)."""
    st = Setup(4, 3, 1500, seed=16)
    rng = np.random.default_rng(16)
    n1 = (st.n + 1) ** 2
    T = np.array([st.T, st.T]); C = np.array([st.C, st.C * np.where(np.arange(n1) >= st.n * (st.n + 1), 2.0, 1.0)])
    group = rng.integers(0, 2, st.y.shape[0]).astype(np.int32)
    keys = np.array([41, 2 ** 33 + 5], dtype=np.uint64)
    starts = st.theta[None, :] * np.array([[1.2], [0.9]])
    eng = st.engine(keys[0], visits=False)
    eng.set_groups(T, C, group)
    eng.set_chains(2, keys)
    eng.set_stage_visits(st.E, st.off, st.t, st.stage, alpha=st.alpha)
    eng.set_chain_theta(starts, next_iter=1)
    eng.set_pi(st.pi, st.beta)
    got = eng.run_chains(8), eng.chain_pi_rows(8), eng.emission_rows(8)
    zbits = eng.zbits
    eng.close()
    for c in range(2):
        want = pm.gibbs_misclass(int(keys[c]), 9, st.n, np.full(st.m, 2.0), np.full(st.m, 2.0), T, C, st.y, st.cens, st.off,
                                 st.t, st.stage, st.E, starts[c], zbits, u=st.u, pi=st.pi, beta=st.beta, alpha=st.alpha,
                                 group=group)
        for g, w in zip(got, want):
            assert np.array_equal(g[c], w[1:])


@pytest.mark.parametrize("graph", [True, False])
def test_set_emission_keeps_each_chains_own_E(graph):
    """set_emission between runs of 3 chains: a new prior with E left as drawn (None), a new E with no prior, then the
    prior back; every chain stays bit for bit the single-chain engine with its key making the same calls."""
    st = Setup(4, 3, 1500, seed=17)
    keys = np.array([3, 2 ** 41 + 9, 1234], dtype=np.uint64)
    alpha2 = np.where(st.alpha > 0, st.alpha * 2.5 + 0.2, 0.0)
    E2 = _emission(st.n, st.S, np.random.default_rng(99))
    E2 = np.where(st.E > 0, E2 + 0.05, 0.0); E2 /= E2.sum(1, keepdims=True)
    steps = [("run", 4), ("set", (None, alpha2)), ("run", 4), ("set", (E2, None)), ("run", 3), ("set", (None, st.alpha)),
             ("run", 3)]

    eng = st.engine(keys[0], alpha=True, use_graph=graph)
    eng.set_chains(3, keys)
    eng.set_chain_theta(np.repeat(st.theta[None], 3, 0), next_iter=1)
    prior, got = True, []
    for what, arg in steps:
        if what == "set":
            eng.set_emission(*arg)
            prior = arg[1] is not None
            continue
        got.append((eng.run_chains(arg), eng.emission_rows(arg) if prior else None))
    eng.close()
    assert not np.array_equal(got[1][1][0], got[1][1][1])          # the chains' E stay their own after set_emission(None, .)
    for c in range(3):
        one = st.engine(keys[c], alpha=True, use_graph=graph)
        one.set_theta(st.theta, next_iter=1)
        prior, r = True, 0
        for what, arg in steps:
            if what == "set":
                one.set_emission(*arg)
                prior = arg[1] is not None
                continue
            assert np.array_equal(got[r][0][c], one.run(arg))
            if prior:
                assert np.array_equal(got[r][1][c], one.emission_rows(arg)[0])
            r += 1
        one.close()


def _indicator_pair(config):
    """Two engines on the same data: stage visits through the 0/1 indicator E of the stages {0, 1}, {2, 3}, and the same
    visits as stage masks; config adds chains and groups, or delayed entry (with the interval bounds every Setup has)."""
    import phasetype_b200 as pb
    st = Setup(4, 2, 1500, seed=15)
    rng = np.random.default_rng(15)
    E = np.array([[1.0, 0.0], [1.0, 0.0], [0.0, 1.0], [0.0, 1.0]])
    masks = synth.stage_masks([0, 0, 1, 1])[st.stage]
    n1 = (st.n + 1) ** 2
    T = np.array([st.T, st.T]); C = np.array([st.C, st.C * np.where(np.arange(n1) >= st.n * (st.n + 1), 2.0, 1.0)])
    group = rng.integers(0, 2, st.y.shape[0]).astype(np.int32)
    first = np.array([st.t[st.off[k]] if st.off[k + 1] > st.off[k] else st.y[k] for k in range(st.y.shape[0])])
    a = np.where(rng.random(st.y.shape[0]) < 0.5, first * rng.uniform(0.0, 1.0, st.y.shape[0]), 0.0)
    sy = st.sy + float(a.sum())
    engs = []
    for stages in (True, False):
        eng = pb.Engine(st.n, st.T, st.C, np.full(st.m, 2.0), np.full(st.m, 2.0), st.y, st.cens, method=METHOD_UNIF, seed=23,
                        sum_y_global=sy)
        eng.set_upper(st.u)
        eng.set_pi(st.pi)
        if config == "chains_groups":
            eng.set_groups(T, C, group)
            eng.set_chains(2)
        if stages:
            eng.set_stage_visits(E, st.off, st.t, st.stage)
        else:
            eng.set_visits(st.off, st.t, masks)
        if config == "entry":
            eng.set_entry(a)
        engs.append(eng)
    return st, engs


@pytest.mark.parametrize("config", ["plain", "chains_groups", "entry"])
def test_indicator_E_equals_the_stage_masks(config):
    st, engs = _indicator_pair(config)
    out = []
    for eng in engs:
        eng.set_theta(st.theta, next_iter=3)
        paths = eng.paths()
        eng.set_chain_theta(np.repeat(st.theta[None], eng.chains, 0), next_iter=1)
        eng.set_pi(st.pi, st.beta)
        out.append(paths + (eng.run_chains(5), eng.chain_pi_rows(5)))
        eng.close()
    for g, w in zip(*out):
        assert np.array_equal(g, w)


def test_observations_without_visits_are_the_plain_engine():
    st = Setup(4, 3, 2000, seed=8)
    plain = st.engine(55, visits=False)
    plain.set_theta(st.theta, next_iter=2)
    Bp, Np, zp = plain.paths()
    plain.set_theta(st.theta, next_iter=1)
    want = plain.run(6)
    plain.close()
    eng = st.engine(55)
    eng.set_theta(st.theta, next_iter=2)
    B, N, z = eng.paths()
    free = np.diff(st.off) == 0
    assert np.array_equal(B[free], Bp[free]) and np.array_equal(N[free], Np[free]) and np.array_equal(z[free], zp[free])
    for how in ("empty", "none", "masks_none"):           # no visits at all, a clear, and masks replacing stages then a clear
        if how == "empty":
            eng.set_stage_visits(st.E, np.zeros(st.y.shape[0] + 1, dtype=np.int64), np.zeros(0), np.zeros(0, dtype=np.uint32))
        elif how == "none":
            eng.set_stage_visits(st.E, st.off, st.t, st.stage)
            eng.set_stage_visits(None, None)
        else:
            eng.set_stage_visits(st.E, st.off, st.t, st.stage, alpha=st.alpha)
            eng.set_visits(st.off, st.t, np.full(st.t.shape[0], (1 << st.n) - 1, dtype=np.uint32))
            assert eng.stages == 0
            with pytest.raises(EngineError, match="stage visits"):
                eng.emission()
            eng.set_visits(None)
        eng.set_theta(st.theta, next_iter=1)
        assert np.array_equal(eng.run(6), want)
    eng.close()


def test_recovery_of_a_misread_progressive_coxian():
    """A 3-phase progressive Coxian (0 -> 1 at a, 1 -> 2 at b, exit from 2 at c, exits from 0 and 1 at e) read in 3 stages,
    each phase as its own stage but 10 % of the readings in an adjacent stage; 2e4 units inspected every 0.4 with exact
    absorption.  The posterior means of theta and of E's free entries fall within 10 % of the truth, and the readings,
    which regress now and then, are refused as stage masks."""
    import phasetype_b200 as pb
    n = 3
    truth = np.array([1.0, 0.8, 1.2, 0.3])               # a, b, c, e
    R = np.diag(truth[:2], 1); s = np.array([truth[3], truth[3], truth[2]])
    E = np.array([[0.9, 0.1, 0.0], [0.1, 0.8, 0.1], [0.0, 0.1, 0.9]])
    T = np.zeros((n + 1, n + 1), dtype=np.int32)
    T[0, 1] = 1; T[1, 2] = 2; T[2, n] = 3; T[0, n] = T[1, n] = 4
    T = T.ravel(order="F"); C = np.ones((n + 1) ** 2)
    rng = np.random.default_rng(2027)
    y, cens, off, t, stage, phase = synth.misclassified_panel(R, s, 20_000, 0.4, 60, E, rng)
    m = truth.shape[0]
    eng = pb.Engine(n, T, C, np.full(m, 1.0), np.full(m, 0.1), y, cens, method=METHOD_UNIF, seed=5, sum_y_global=float(y.sum()))
    with pytest.raises(EngineError, match="cannot produce"):
        eng.set_visits(off, t, (1 << stage.astype(np.int64)).astype(np.uint32))
    alpha = np.where(E > 0, 1.0, 0.0)
    start = np.array([[0.8, 0.2, 0.0], [0.2, 0.6, 0.2], [0.0, 0.2, 0.8]])
    eng.set_stage_visits(start, off, t, stage, alpha=alpha)
    eng.set_chains(4)
    eng.set_chain_theta(truth[None, :] * rng.uniform(0.7, 1.4, (4, m)), next_iter=1)
    draws = eng.run_chains(600)[:, 150:, :]
    Es = eng.emission_rows(600)[:, 150:]
    eng.close()
    th = draws.reshape(-1, m).mean(0)
    assert (np.abs(th - truth) < 0.1 * truth).all(), (th, truth)
    free = alpha > 0
    Em = Es.reshape(-1, n, n).mean(0)
    assert (np.abs(Em[free] - E[free]) < 0.1 * E[free]).all(), (Em, E)


def test_refusals_leave_the_engine_as_it_was():
    import phasetype_b200 as pb
    st = Setup(4, 3, 300, seed=14)
    l = st.y.shape[0]
    eng = st.engine(17, alpha=True)
    eng.set_theta(st.theta, next_iter=3)
    before = eng.paths(), eng.emission()

    def same():
        after = eng.paths(), eng.emission()
        assert all(np.array_equal(a, b) for a, b in zip(after[0], before[0])) and np.array_equal(after[1], before[1])

    def refused(what, E=st.E, off=st.off, t=st.t, stage=st.stage, alpha=st.alpha):
        with pytest.raises(EngineError, match=what):
            eng.set_stage_visits(E, off, t, stage, alpha=alpha)
        same()

    refused("stages = 33", E=np.full((4, MAX_STAGES + 1), 1.0 / (MAX_STAGES + 1)), alpha=None)
    bad = st.stage.copy(); bad[0] = 3
    refused("not below stages", stage=bad)
    bad = st.E.copy(); bad[1, 0] = -0.1; bad[1, 1] += 0.1
    refused("not a probability", E=bad, alpha=None)
    bad = st.E.copy(); bad[2, 0] = np.nan
    refused("not a probability", E=bad, alpha=None)
    bad = st.E.copy(); bad[0] *= 1.0 + 1e-9
    refused("not 1", E=bad, alpha=None)
    bad = st.alpha.copy(); bad[bad > 0] = -1.0
    refused("not negative", alpha=bad)
    bad = st.alpha.copy(); bad[st.E > 0] = 0.05
    refused("below 0.1", alpha=bad)
    bad = st.alpha.copy(); bad[0, :] = 1.0
    refused("support", alpha=bad)
    k = int(np.flatnonzero((np.diff(st.off) >= 2) & (st.y > 0))[0])
    bad = st.t.copy(); bad[st.off[k] + 1] = bad[st.off[k]]
    refused("must increase", t=bad)
    cnt = np.zeros(l, dtype=np.int64); j = int(np.argmax(st.y)); cnt[j] = MAX_VISITS + 1
    refused("PHT_MAX_VISITS", off=np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64),
            t=np.linspace(0.0, st.y[j], MAX_VISITS + 1), stage=np.zeros(MAX_VISITS + 1, dtype=np.uint32))
    with pytest.raises(EngineError, match="not 1"):
        eng.set_emission(np.full((4, 3), 0.5), None)
    with pytest.raises(EngineError, match="support"):
        eng.set_emission(None, np.ones((4, 3)))
    same()
    eng.close()
    # a reading sequence no path can produce: a Coxian whose phase 2 is always read as stage 2 cannot be read as stage 0
    # after it; E, pi and structures that would make the engine's readings impossible are refused while they are set
    n = 3
    Tc = np.zeros((n + 1, n + 1), dtype=np.int32); Tc[0, 1] = 1; Tc[1, 2] = 2; Tc[2, n] = 3; Tc = Tc.ravel(order="F")
    yc = np.array([2.0, 2.0]); cc = np.array([0, 1], dtype=np.int32)
    E = np.array([[0.9, 0.1, 0.0], [0.1, 0.9, 0.0], [0.0, 0.0, 1.0]])
    eng = pb.Engine(n, Tc, np.ones((n + 1) ** 2), np.full(3, 2.0), np.full(3, 2.0), yc, cc, method=METHOD_UNIF, seed=1)
    offc = np.array([0, 2, 2], dtype=np.int64)
    with pytest.raises(EngineError, match="cannot produce"):
        eng.set_stage_visits(E, offc, np.array([0.5, 1.0]), np.array([2, 0], dtype=np.uint32))
    eng.set_stage_visits(E, offc, np.array([0.0, 1.5]), np.array([1, 0], dtype=np.uint32))    # phase 0 read as 1, then 0
    eng.set_theta(np.ones(3), next_iter=2)
    before = eng.paths(), eng.emission()
    with pytest.raises(EngineError, match="cannot produce"):        # stage 1 then impossible at t = 0 (pi = e1)
        eng.set_emission(np.array([[1.0, 0.0, 0.0], [0.1, 0.9, 0.0], [0.0, 0.0, 1.0]]), None)
    with pytest.raises(EngineError, match="cannot produce"):        # a pi that cannot start where stage 1 is read
        eng.set_pi(np.array([0.0, 0.0, 1.0]))
    with pytest.raises(EngineError, match="cannot absorb"):         # a structure with no way out of phase 0: no exit
        Cz = np.ones((n + 1, n + 1)); Cz[0, 1] = 0.0
        eng.set_groups(Tc[None], Cz.ravel(order="F")[None], np.zeros(2, dtype=np.int32))
    assert np.array_equal(eng.get_pi(), np.eye(n)[0]) and np.array_equal(eng.emission(), before[1])
    assert all(np.array_equal(a, b) for a, b in zip(eng.paths(), before[0]))
    with pytest.raises(EngineError, match="not being inferred"):
        eng.emission_rows(1)
    # counts, in either order
    with pytest.raises(EngineError, match="visits"):
        eng.set_counts(np.array([1, 1], dtype=np.uint32))
    eng.set_stage_visits(None, None)
    with pytest.raises(EngineError, match="stage visits"):
        eng.set_emission(E, None)
    eng.set_counts(np.array([1, 2], dtype=np.uint32))
    with pytest.raises(EngineError, match="counts"):
        eng.set_stage_visits(E, offc, np.array([0.0, 1.5]), np.array([1, 0], dtype=np.uint32))
    eng.close()
    # methods other than 64; several ranks
    wl = synth.config(1, l=50)
    E1 = np.full((wl.n, 2), 0.5)
    other = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=1, seed=1)
    with pytest.raises(EngineError, match="method 64"):
        other.set_stage_visits(E1, np.zeros(51, dtype=np.int64), np.zeros(0), np.zeros(0, dtype=np.uint32))
    other.close()
    two = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y[::2], wl.censored[::2], method=METHOD_UNIF, seed=1, rank=0, world=2,
                    zbits=30)
    with pytest.raises(EngineError, match="world = 1"):
        two.set_stage_visits(E1, np.zeros(two.l_local + 1, dtype=np.int64), np.zeros(0), np.zeros(0, dtype=np.uint32))
    two.close()
