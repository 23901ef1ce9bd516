"""Panel observations (pht_engine_set_visits) on the GPU: every panel path equals the host build (oracle/pht_oracle_panel.c)
bit for bit; a chain equals the host chain; observations without visits draw the plain engine's paths; chains, groups,
delayed entry and graph launches keep their contracts; 8 chains recover a Coxian observed in two stages; and the
refusals, each leaving the engine as it was."""
import numpy as np
import pytest

from oracle import pyoracle_panel as pp
from phasetype_b200 import synth
from phasetype_b200._lib import MAX_VISITS, METHOD_UNIF, EngineError
from phasetype_b200.diagnostics import split_rhat
from tests import util

pytestmark = pytest.mark.gpu


def _data(n, l, rng, frac=0.6, singletons=False):
    """Exact, right-, interval- and left-censored observations of a dense model; a share frac of them (y > 0) with 1..5
    visits at sorted times in [0, y] (some at 0 and at y), masks random non-empty phase sets (or single phases)."""
    y = rng.exponential(1.0, l) + 0.01
    kind = rng.integers(0, 4, l)
    cens = (kind > 0).astype(np.int32)
    y = np.where(kind == 3, 0.0, y)
    u = np.where(kind >= 2, y + rng.exponential(0.7, l) + 1e-3, np.inf)
    offs, ts, ms = [0], [], []
    full = (1 << n) - 1
    for k in range(l):
        m = 0
        if y[k] == 0.0:
            if rng.random() < 0.3:
                ts.append(0.0); ms.append(int(rng.integers(1, full + 1))); m = 1
        elif rng.random() < frac:
            m = int(rng.integers(1, 6))
            t = np.sort(rng.uniform(0.0, y[k], m))
            if rng.random() < 0.2:
                t[0] = 0.0
            if rng.random() < 0.2:
                t[-1] = y[k]
            t = np.unique(t); m = t.shape[0]
            ts.extend(t.tolist())
            for _ in range(m):
                ms.append(1 << int(rng.integers(0, n)) if singletons else int(rng.integers(1, full + 1)))
        offs.append(offs[-1] + m)
    return y, cens, u, np.array(offs, dtype=np.int64), np.array(ts), np.array(ms, dtype=np.uint32)


class Setup:
    def __init__(self, n, l, seed, singletons=False):
        rng = np.random.default_rng(seed)
        self.n = n
        R, s = util.dense_rates(n, rng)
        self.T, self.C, self.theta = util.general_model(R, s)
        self.m = self.theta.shape[0]
        self.y, self.cens, self.u, self.off, self.t, self.mask = _data(n, l, rng, singletons=singletons)
        self.pi = rng.uniform(0.1, 1.0, n); self.pi /= self.pi.sum()
        self.beta = rng.uniform(0.5, 2.0, n)
        self.sy = float(np.where(np.isfinite(self.u), self.u, self.y).sum())

    def engine(self, seed, visits=True, **kw):
        import phasetype_b200 as pb
        eng = pb.Engine(self.n, self.T, self.C, np.full(self.m, 2.0), np.full(self.m, 2.0), self.y, self.cens,
                        method=METHOD_UNIF, seed=int(seed), sum_y_global=self.sy, **kw)
        eng.set_upper(self.u)
        eng.set_pi(self.pi)                           # visits at t = 0 need a start distribution that can begin in their masks
        if visits:
            eng.set_visits(self.off, self.t, self.mask)
        return eng


def _oracle_paths(st, eng, seed, it):
    mdl = eng.model()
    B, N, z, err = pp.panel_paths(seed, it, st.y, st.cens, st.off, st.t, st.mask, mdl["S"], mdl["s"], u=st.u, pi=st.pi)
    assert err == 0
    return B, N, z


@pytest.mark.parametrize("n", [1, 4, 8, 32])
@pytest.mark.parametrize("singletons", [False, True])
def test_paths_equal_the_host_build(n, singletons):
    st = Setup(n, 1200 if n <= 8 else 300, seed=40 + n, singletons=singletons)
    eng = st.engine(91)
    eng.set_theta(st.theta, next_iter=5)
    eng.set_pi(st.pi)
    got = eng.paths()
    want = _oracle_paths(st, eng, 91, 5)
    eng.close()
    for g, w in zip(got, want):
        assert np.array_equal(g, w)


def test_chain_equals_host_chain():
    st = Setup(4, 1500, seed=7)
    start = st.theta * 1.3
    eng = st.engine(31)
    eng.set_theta(start, next_iter=1)
    eng.set_pi(st.pi, st.beta)
    got = eng.run(20)
    pis = eng.pi_rows(20)
    zbits = eng.zbits
    eng.close()
    want, wpi = pp.gibbs_panel(31, 21, st.n, np.full(st.m, 2.0), np.full(st.m, 2.0), st.T, st.C, st.y, st.cens, st.off, st.t,
                               st.mask, start, zbits, u=st.u, pi=st.pi, beta=st.beta)
    assert np.array_equal(got, want[1:]) and np.array_equal(pis, wpi[1:])


def test_observations_without_visits_are_the_plain_engine():
    st = Setup(4, 2000, seed=8)
    plain = st.engine(55, visits=False)
    plain.set_theta(st.theta, next_iter=2)
    Bp, Np, zp = plain.paths()
    plain.set_theta(st.theta, next_iter=1)
    plain.set_pi(st.pi, st.beta)
    want = plain.run(8), plain.pi_rows(8)
    plain.close()
    eng = st.engine(55)
    eng.set_theta(st.theta, next_iter=2)
    B, N, z = eng.paths()
    free = np.diff(st.off) == 0
    assert np.array_equal(B[free], Bp[free]) and np.array_equal(N[free], Np[free]) and np.array_equal(z[free], zp[free])
    # all-empty visits, and set_visits(None), give the plain engine's chain
    for how in ("empty", "none"):
        if how == "empty":
            eng.set_visits(np.zeros(st.y.shape[0] + 1, dtype=np.int64), np.zeros(0), np.zeros(0, dtype=np.uint32))
        else:
            eng.set_visits(st.off, st.t, st.mask)
            eng.set_visits(None)
        eng.set_theta(st.theta, next_iter=1)
        eng.set_pi(st.pi, st.beta)
        got = eng.run(8), eng.pi_rows(8)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    eng.close()


def test_chains_equal_single_chain_engines():
    st = Setup(4, 1500, seed=9)
    keys = np.array([11, 2 ** 40 + 3, 77], dtype=np.uint64)
    thetas = st.theta[None, :] * np.array([[0.8], [1.0], [1.3]])
    eng = st.engine(keys[0])
    eng.set_chains(3, keys)                           # visits first, chains after
    eng.set_chain_theta(thetas, next_iter=1)
    eng.set_pi(st.pi, st.beta)
    got = eng.run_chains(6), eng.chain_pi_rows(6)
    eng.close()
    for c in range(3):
        one = st.engine(keys[c])
        one.set_theta(thetas[c], next_iter=1)
        one.set_pi(st.pi, st.beta)
        assert np.array_equal(got[0][c], one.run(6)) and np.array_equal(got[1][c], one.pi_rows(6))
        one.close()


def test_groups_paths_are_each_groups_own():
    st = Setup(4, 1500, seed=10)
    rng = np.random.default_rng(10)
    n1 = (st.n + 1) ** 2
    T = np.array([st.T, st.T]); C = np.array([st.C, st.C * np.where(np.arange(n1) >= st.n * (st.n + 1), 2.0, 1.0)])
    group = rng.integers(0, 2, st.y.shape[0]).astype(np.int32)
    eng = st.engine(21, visits=False)
    eng.set_groups(T, C, group)
    eng.set_visits(st.off, st.t, st.mask)             # groups first, visits after
    eng.set_theta(st.theta, next_iter=4)
    eng.set_pi(st.pi)
    B, N, z = eng.paths()
    Ng, Bg, zg = eng.group_stats()
    eng.close()
    for g in range(2):
        import phasetype_b200 as pb
        one = pb.Engine(st.n, T[g], C[g], np.full(st.m, 2.0), np.full(st.m, 2.0), st.y, st.cens, method=METHOD_UNIF, seed=21,
                        sum_y_global=st.sy)
        one.set_upper(st.u)
        one.set_pi(st.pi)
        one.set_visits(st.off, st.t, st.mask)
        one.set_theta(st.theta, next_iter=4)
        one.set_pi(st.pi)
        Bo, No, zo = one.paths()
        one.close()
        sel = group == g
        assert np.array_equal(B[sel], Bo[sel]) and np.array_equal(N[sel], No[sel]) and np.array_equal(z[sel], zo[sel])
        assert np.array_equal(Ng[g], N[sel].astype(np.int64).sum(0)) and np.array_equal(Bg[g], np.bincount(B[sel], minlength=st.n))


def test_delayed_entry_ghosts_do_not_depend_on_visits():
    st = Setup(4, 1500, seed=12)
    rng = np.random.default_rng(12)
    first = np.array([st.t[st.off[k]] if st.off[k + 1] > st.off[k] else st.y[k] for k in range(st.y.shape[0])])
    a = np.where(rng.random(st.y.shape[0]) < 0.5, first * rng.uniform(0.0, 1.0, st.y.shape[0]), 0.0)
    a = np.where(rng.random(st.y.shape[0]) < 0.1, first, a)      # a visit at the entry age itself
    a = np.minimum(a, st.y)
    sy = st.sy + float(a.sum())
    import phasetype_b200 as pb
    outs = []
    for order in ("none", "entry_first", "visits_first"):
        eng = pb.Engine(st.n, st.T, st.C, np.full(st.m, 2.0), np.full(st.m, 2.0), st.y, st.cens, method=METHOD_UNIF, seed=5,
                        sum_y_global=sy)
        eng.set_upper(st.u)
        eng.set_pi(st.pi)
        if order == "visits_first":
            eng.set_visits(st.off, st.t, st.mask)
        eng.set_entry(a)
        if order == "entry_first":
            eng.set_visits(st.off, st.t, st.mask)
        eng.set_theta(st.theta, next_iter=2)
        outs.append(eng.entry_paths())
        if order != "none":
            eng.set_theta(st.theta, next_iter=1)
            outs.append(eng.run(4))
        eng.close()
    for g, w in zip(outs[1], outs[0]):
        assert np.array_equal(g, w)
    for g, w in zip(outs[3], outs[0]):
        assert np.array_equal(g, w)
    assert np.array_equal(outs[2], outs[4])


def test_graph_equals_direct_launches():
    st = Setup(8, 3000, seed=13)
    rows = []
    for graph in (True, False):
        eng = st.engine(3, use_graph=graph)
        eng.set_chains(2)
        eng.set_chain_theta(np.array([st.theta, st.theta * 1.2]), next_iter=1)
        eng.set_pi(st.pi, st.beta)
        rows.append((eng.run_chains(6), eng.chain_pi_rows(6)))
        eng.close()
    assert np.array_equal(rows[0][0], rows[1][0]) and np.array_equal(rows[0][1], rows[1][1])


def test_recovery_of_a_coxian_seen_in_two_stages():
    """A 4-phase Coxian seen in two stages of two phases each, 1e5 units inspected every 0.5 with exact absorption: 8
    chains mix (split R-hat < 1.01) and every posterior mean lies within 4 posterior SDs of the truth.  Each stage is
    Erlang-like (stage 0: rate a for 0 -> 1 and 1 -> 2; stage 1: rate c for 2 -> 3 and for the exit from 3), with the exit
    rate e from phases 0..2.  Untied rates inside a stage are not identified: with a' for 0 -> 1 and b' for 1 -> 2 the
    law of the stage process is the same under a' <-> b', and with c' for 2 -> 3 and d' for the exit from 3 the same
    under (c', d') -> (d' - e, c' + e), so the posterior has no single truth to recover."""
    import phasetype_b200 as pb
    n = 4
    truth = np.array([1.4, 1.1, 0.2])                   # a, c, e
    R = np.diag([truth[0], truth[0], truth[1]], 1); s = np.array([truth[2]] * 3 + [truth[1]])
    T = np.zeros((n + 1, n + 1), dtype=np.int32)
    T[0, 1] = T[1, 2] = 1; T[2, 3] = T[3, n] = 2
    T[0, n] = T[1, n] = T[2, n] = 3
    T = T.ravel(order="F"); C = np.ones((n + 1) ** 2)
    rng = np.random.default_rng(2026)
    y, cens, off, t, mask = synth.panel(R, s, 100_000, 0.5, 40, [0, 0, 1, 1], rng)
    m = truth.shape[0]
    eng = pb.Engine(n, T, C, np.full(m, 1.0), np.full(m, 0.1), y, cens, method=METHOD_UNIF, seed=99, sum_y_global=float(y.sum()))
    eng.set_visits(off, t, mask)
    eng.set_chains(8)
    eng.set_chain_theta(truth[None, :] * rng.uniform(0.6, 1.6, (8, m)), next_iter=1)
    draws = eng.run_chains(1500)[:, 300:, :]
    eng.close()
    assert split_rhat(draws).max() < 1.01
    flat = draws.reshape(-1, m)
    assert (np.abs(flat.mean(0) - truth) < 4.0 * flat.std(0)).all(), (flat.mean(0), flat.std(0), truth)


def test_refusals_leave_the_engine_as_it_was():
    import phasetype_b200 as pb
    st = Setup(4, 300, seed=14)
    l = st.y.shape[0]
    eng = st.engine(17)
    eng.set_theta(st.theta, next_iter=3)
    before = eng.paths()

    def refused(off, t, mask, what):
        with pytest.raises(EngineError, match=what):
            eng.set_visits(off, t, mask)
        after = eng.paths()
        assert all(np.array_equal(a, b) for a, b in zip(after, before))

    k = int(np.flatnonzero((np.diff(st.off) >= 2) & (st.y > 0))[0])
    bad_t = st.t.copy(); bad_t[st.off[k] + 1] = bad_t[st.off[k]]
    refused(st.off, bad_t, st.mask, "must increase")
    bad_t = st.t.copy(); bad_t[st.off[k]] = -1.0
    refused(st.off, bad_t, st.mask, "negative")
    bad_t = st.t.copy(); bad_t[st.off[k + 1] - 1] = st.y[k] * 1.5 + 0.1
    refused(st.off, bad_t, st.mask, "above y")
    bad_m = st.mask.copy(); bad_m[st.off[k]] = 0
    refused(st.off, st.t, bad_m, "empty mask")
    bad_m = st.mask.copy(); bad_m[st.off[k]] = 1 << 4
    refused(st.off, st.t, bad_m, "at or above n")
    # y = 0: only a single visit at t = 0
    z0 = int(np.flatnonzero(st.y == 0.0)[0])
    cnt = np.zeros(l, dtype=np.int64); cnt[z0] = 2
    off2 = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    t2 = np.zeros(off2[-1]); m2 = np.full(off2[-1], 1, dtype=np.uint32)
    refused(off2, t2, m2, "y = 0")
    # too many visits
    cnt = np.zeros(l, dtype=np.int64); j = int(np.argmax(st.y)); cnt[j] = MAX_VISITS + 1
    off3 = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    refused(off3, np.linspace(0.0, st.y[j], MAX_VISITS + 1), np.full(MAX_VISITS + 1, 1, dtype=np.uint32), "PHT_MAX_VISITS")
    eng.close()
    # a visit sequence the structure cannot produce: a Coxian cannot go back from phase 2 to phase 0
    n = 3
    Tc = np.zeros((n + 1, n + 1), dtype=np.int32); Tc[0, 1] = 1; Tc[1, 2] = 2; Tc[2, n] = 3; Tc = Tc.ravel(order="F")
    yc = np.array([2.0, 2.0]); cc = np.array([0, 1], dtype=np.int32)
    eng = pb.Engine(n, Tc, np.ones((n + 1) ** 2), np.full(3, 2.0), np.full(3, 2.0), yc, cc, method=METHOD_UNIF, seed=1)
    offc = np.array([0, 2, 2], dtype=np.int64)
    with pytest.raises(EngineError, match="cannot produce"):
        eng.set_visits(offc, np.array([0.5, 1.0]), np.array([1 << 2, 1 << 0], dtype=np.uint32))
    with pytest.raises(EngineError, match="cannot absorb"):        # exact at t = y in phase 0, which has no exit
        eng.set_visits(offc, np.array([0.5, 2.0]), np.array([1 << 0, 1 << 0], dtype=np.uint32))
    with pytest.raises(EngineError, match="cannot produce"):        # seen in phase 1 at t = 0, but pi = e1 starts in phase 0
        eng.set_visits(offc, np.array([0.0, 1.5]), np.array([1 << 1, 1 << 1], dtype=np.uint32))
    eng.set_visits(offc, np.array([0.0, 1.5]), np.array([1 << 0, 1 << 1], dtype=np.uint32))   # possible
    eng.set_theta(np.ones(3), next_iter=2)
    before = eng.paths()
    with pytest.raises(EngineError, match="cannot produce"):        # a pi that cannot start in phase 0, seen at t = 0
        eng.set_pi(np.array([0.0, 1.0, 0.0]))
    with pytest.raises(EngineError, match="cannot produce"):        # a structure with no way from phase 0 to phase 1
        Cz = np.ones((n + 1, n + 1)); Cz[0, 1] = 0.0
        eng.set_groups(Tc[None], Cz.ravel(order="F")[None], np.zeros(2, dtype=np.int32))
    assert np.array_equal(eng.get_pi(), np.eye(n)[0])
    assert all(np.array_equal(a, b) for a, b in zip(eng.paths(), before))
    # counts, in either order
    with pytest.raises(EngineError, match="visits"):
        eng.set_counts(np.array([1, 1], dtype=np.uint32))
    eng.set_visits(None)
    eng.set_counts(np.array([1, 2], dtype=np.uint32))
    with pytest.raises(EngineError, match="counts"):
        eng.set_visits(offc, np.array([0.5, 1.5]), np.array([1 << 0, 1 << 1], dtype=np.uint32))
    eng.close()
    # methods other than 64; several ranks
    wl = synth.config(1, l=50)
    other = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=1, seed=1)
    with pytest.raises(EngineError, match="method 64"):
        other.set_visits(np.zeros(51, dtype=np.int64), np.zeros(0), np.zeros(0, dtype=np.uint32))
    other.close()
    two = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y[::2], wl.censored[::2], method=METHOD_UNIF, seed=1, rank=0, world=2,
                    zbits=30)
    with pytest.raises(EngineError, match="world = 1"):
        two.set_visits(np.zeros(two.l_local + 1, dtype=np.int64), np.zeros(0), np.zeros(0, dtype=np.uint32))
    two.close()
