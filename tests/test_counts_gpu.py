"""Observations with counts (method 64, pht_engine_set_counts) on the GPU: an engine with counts is, bit for bit, the
engine created on the expanded data np.repeat(records, counts) -- sweep statistics, theta and pi rows, with chains and
groups in either order of the calls, through graph replays and direct launches; all-ones counts and clearing the counts
give the engine without counts; a record just under 2^32 units checks the 32-bit index and the counter flush; and the
refusals."""
import numpy as np
import pytest

from phasetype_b200._lib import METHOD_UNIF, EngineError
from tests import util

pytestmark = pytest.mark.gpu

THRESHOLD, CHUNK = 8, 64            # small, so that every split of a record is exercised (results do not depend on them)


@pytest.fixture(autouse=True)
def _small_split(monkeypatch):
    monkeypatch.setenv("PHT_B200_COUNTS_THRESHOLD", str(THRESHOLD))
    monkeypatch.setenv("PHT_B200_COUNTS_CHUNK", str(CHUNK))


def _zbits(y, u, w):
    import phasetype_b200 as pb
    return int(pb.lib().pht_choose_zbits(float((np.where(np.isfinite(u), u, y) * w).sum())))


class Setup:
    """l records of every kind (exact, right-, interval-, left-censored) with counts 0, 1, just below, at and above the
    threshold, and one record spanning many chunks."""

    def __init__(self, n, l, seed, groups=1):
        rng = np.random.default_rng(seed)
        self.n = n
        R, s = util.dense_rates(n, rng)
        self.T, self.C, self.theta = util.general_model(R, s)
        self.m = self.theta.shape[0]
        y = rng.exponential(1.0, l) + 0.01
        kind = rng.integers(0, 4, l)
        self.cens = (kind > 0).astype(np.int32)
        self.y = np.where(kind == 3, 0.0, y)
        self.u = np.where(kind >= 2, self.y + rng.exponential(0.7, l) + 1e-3, np.inf)
        w = rng.choice(np.array([0, 1, 2, THRESHOLD - 1, THRESHOLD, THRESHOLD + 1, 3 * THRESHOLD]), l)
        w[rng.integers(0, l)] = 7 * CHUNK + 5
        self.w = w.astype(np.uint32)
        self.group = rng.integers(0, groups, l).astype(np.int32)
        self.pi = rng.uniform(0.1, 1.0, n); self.pi /= self.pi.sum()
        self.beta = rng.uniform(0.5, 2.0, n)
        self.zbits = _zbits(self.y, self.u, self.w)

    def engine(self, seed, expanded, use_graph=True):
        import phasetype_b200 as pb
        rep = (lambda a: np.repeat(a, self.w)) if expanded else (lambda a: a)
        eng = pb.Engine(self.n, self.T, self.C, np.full(self.m, 2.0), np.full(self.m, 2.0), rep(self.y), rep(self.cens),
                        method=METHOD_UNIF, seed=int(seed), zbits=self.zbits, use_graph=use_graph)
        eng.set_upper(rep(self.u))
        return eng

    def pair(self, seed, **kw):
        a = self.engine(seed, True, **kw)
        b = self.engine(seed, False, **kw)
        b.set_counts(self.w)
        return a, b


def _same_chain(a, b, st, sweeps=20):
    for e in (a, b):
        e.set_theta(st.theta, next_iter=1)
        e.set_pi(st.pi, st.beta)
    sa, sb = a.sweep_stats(), b.sweep_stats()
    for x, y in zip(sa, sb):
        assert np.array_equal(x, y)
    ta, tb = a.run(sweeps), b.run(sweeps)
    assert np.array_equal(ta, tb)
    assert np.array_equal(a.pi_rows(sweeps), b.pi_rows(sweeps))
    return sa


@pytest.mark.parametrize("n", [1, 4, 8, 32])
def test_counts_equal_the_expanded_engine(n):
    st = Setup(n, 300 if n < 32 else 60, seed=n)
    a, b = st.pair(17)
    N, B, z = _same_chain(a, b, st)
    assert B.sum() == st.w.astype(np.int64).sum()
    assert b.counters()["paths"] >= st.w.astype(np.int64).sum()          # every unit drawn, counted as a path
    a.close(); b.close()


def test_default_split(monkeypatch):
    """the library's own threshold and chunk size (the other tests shrink them)"""
    monkeypatch.delenv("PHT_B200_COUNTS_THRESHOLD"); monkeypatch.delenv("PHT_B200_COUNTS_CHUNK")
    st = Setup(4, 200, seed=5)
    st.w[:3] = [100, 5000, 3000]
    st.zbits = _zbits(st.y, st.u, st.w)
    a, b = st.pair(3)
    _same_chain(a, b, st, sweeps=10)
    a.close(); b.close()


def test_all_ones_and_cleared_counts_are_the_plain_engine():
    st = Setup(4, 500, seed=2)
    st.w[:] = 1
    plain = st.engine(9, False)
    ones = st.engine(9, False)
    ones.set_counts(st.w)
    _same_chain(plain, ones, st, sweeps=10)
    cleared = st.engine(9, False)
    cleared.set_counts(np.arange(500) % 5)
    cleared.set_counts(None)
    plain2 = st.engine(9, False)
    _same_chain(plain2, cleared, st, sweeps=10)
    for e in (plain, ones, cleared, plain2):
        e.close()


@pytest.mark.parametrize("order", ["counts_first", "counts_last"])
def test_chains_and_groups(order):
    from tests.test_groups_gpu import _exit_groups
    st = Setup(4, 300, seed=11, groups=3)
    rng = np.random.default_rng(4)
    T, C, theta = _exit_groups(4, 3, rng)
    st.T, st.C, st.theta = T[0], C[0], theta
    st.m = theta.shape[0]
    chains = 3
    keys = np.array([11, 22, 33], dtype=np.uint64)
    thetas = theta[None, :] * rng.uniform(0.5, 2.0, (chains, st.m))

    def setup(e, expanded, counts):
        if counts and order == "counts_first":
            e.set_counts(st.w)
        e.set_chains(chains, keys)
        e.set_groups(T, C, np.repeat(st.group, st.w) if expanded else st.group)
        if counts and order == "counts_last":
            e.set_counts(st.w)
        e.set_chain_theta(thetas, next_iter=1)
        e.set_pi(st.pi, st.beta)

    a = st.engine(keys[0], True); setup(a, True, False)
    b = st.engine(keys[0], False); setup(b, False, True)
    ga, gb = a.group_stats(), b.group_stats()
    for x, y in zip(ga, gb):
        assert np.array_equal(x, y)
    assert np.array_equal(a.run_chains(12), b.run_chains(12))
    assert np.array_equal(a.chain_pi_rows(12), b.chain_pi_rows(12))
    a.close(); b.close()


def test_graph_and_direct_launches_agree():
    st = Setup(8, 200, seed=6)
    g = st.engine(5, False, use_graph=True); g.set_counts(st.w)
    d = st.engine(5, False, use_graph=False); d.set_counts(st.w)
    _same_chain(g, d, st, sweeps=10)
    g.close(); d.close()


def test_counts_just_under_two_to_the_32():
    """one exact record of 2^32 - 2 units at n = 1: N[0,0] and B are the count (every unit is absorbed once)"""
    import phasetype_b200 as pb
    w = np.array([2 ** 32 - 2], dtype=np.uint32)
    y = np.array([0.01])
    zb = _zbits(y, np.array([np.inf]), w)
    T = np.array([0, 0, 1, 0], dtype=np.int32); C = np.ones(4)
    eng = pb.Engine(1, T, C, [2.0], [2.0], y, np.zeros(1, np.int32), method=METHOD_UNIF, seed=3, zbits=zb)
    eng.set_counts(w)
    eng.set_theta([1.0], next_iter=1)
    N, B, z = eng.sweep_stats()
    assert N[0] == 2 ** 32 - 2 and B[0] == 2 ** 32 - 2
    eng.close()


def test_refusals():
    import phasetype_b200 as pb
    st = Setup(3, 100, seed=8)
    w = st.w

    def fresh(**kw):
        return pb.Engine(st.n, st.T, st.C, np.full(st.m, 2.0), np.full(st.m, 2.0), st.y, st.cens,
                         method=kw.pop("method", METHOD_UNIF), seed=1, zbits=kw.pop("zbits", st.zbits), **kw)

    e = fresh(method=1)
    with pytest.raises(EngineError, match="need method 64"):
        e.set_counts(w)
    e.close()
    e = fresh(rank=0, world=2)
    with pytest.raises(EngineError, match="world = 1"):
        e.set_counts(w)
    e.close()
    engs = [fresh(rank=r, world=2) for r in range(2)]
    h = b"".join(x.peer_handle() for x in engs)
    for x in engs:
        x.peer_attach(h)
    with pytest.raises(EngineError, match="exchange windows are attached"):
        engs[0].set_counts(w)
    for x in engs:
        x.close()

    e = fresh()
    e.set_upper(st.u)
    e.set_theta(st.theta, next_iter=2)
    want = e.sweep_stats()

    def unchanged():
        got = e.sweep_stats()
        assert all(np.array_equal(x, y) for x, y in zip(got, want))

    with pytest.raises(EngineError, match="local records"):
        e.set_counts(w[:-1])
    e.set_entry(np.zeros(st.y.shape[0]))
    with pytest.raises(EngineError, match="entry ages"):
        e.set_counts(w)
    e.set_entry(None)
    big = np.full(st.y.shape[0], 2 ** 32 // st.y.shape[0] + 1, dtype=np.uint64)
    with pytest.raises(EngineError, match="2\\^32"):
        e.set_counts(big)
    with pytest.raises(EngineError, match="too fine for these counts"):
        e.set_counts(np.full(st.y.shape[0], 4000, dtype=np.uint32))
    unchanged()

    e.set_counts(w)
    with pytest.raises(EngineError, match="entry ages"):
        e.set_entry(np.zeros(st.y.shape[0]))
    with pytest.raises(EngineError, match="not recorded while counts are set"):
        e.paths(0, 5)
    with pytest.raises(EngineError, match="too fine for these bounds"):
        e.set_upper(np.where(st.cens == 1, st.y + 1e4, np.inf))
    e.set_counts(None)
    unchanged()
    e.close()
