"""Panel observations (method 64 with visits) in the host build of the sampler, oracle/pht_oracle_panel.c: the paths have the
exact conditional law given the start distribution, the visits and the terminal information.  The exact values come from a
forward-backward pass over the visits in numpy (scipy expm per gap) and the Van Loan integrals of tests/test_unif_oracle.py
per gap; the tolerances from the Monte Carlo standard errors of ~2e5 host draws."""
import numpy as np
import pytest
import scipy.linalg as sl

from oracle import pyoracle_panel as pp
from tests import test_unif_oracle as tu
from tests import util

DRAWS = 200_000
STAGES_COX = (0b0011, 0b1100)           # the tied Coxian's two clinical stages of two phases each


def _vanloan(Sm, i, k, d):
    n = Sm.shape[0]
    E = np.zeros((n, n)); E[i, k] = 1.0
    return sl.expm(np.block([[Sm, E], [np.zeros((n, n)), Sm]]) * d)[:n, n:]


def _full(Sm, s, p):
    """Total statistics of the unconditioned chain from the (unnormalised) start weights p: z, N (off-diagonal), exits."""
    occ = p @ np.linalg.inv(-Sm)
    return occ, occ[:, None] * Sm * (1 - np.eye(s.shape[0])), occ * s


def panel_expectations(Sm, s, pi, y, kind, vt, vm, u=None):
    """Exact E[z], E[N_ij] (i != j), E[exits], P(start = a) and P(x_j = c) of a panel path."""
    n = s.shape[0]
    ind = [np.array([(mk >> c) & 1 for c in range(n)], dtype=float) for mk in vm]
    times = [0.0] + list(vt) + [y]
    gaps = np.diff(times)
    m = len(vt)
    if kind == "exact":
        v = s.copy()
    elif kind == "right":
        v = np.ones(n)
    else:
        v = 1.0 - sl.expm(Sm * (u - y)) @ np.ones(n)
    E = [sl.expm(Sm * g) for g in gaps]
    beta = [None] * (m + 2)                          # beta[j]: weights at t_j including the mask of visit j; beta[m+1] = v
    beta[m + 1] = v
    for j in range(m, 0, -1):
        beta[j] = ind[j - 1] * (E[j] @ beta[j + 1])
    beta[0] = E[0] @ beta[1]
    alpha = [pi.astype(float)]                       # alpha[j]: forward weights at t_j including the mask of visit j
    for j in range(1, m + 1):
        alpha.append((alpha[j - 1] @ E[j - 1]) * ind[j - 1])
    alpha.append(alpha[m] @ E[m])
    Z = pi @ beta[0]
    xs = [alpha[j] * (E[j] @ beta[j + 1]) / Z for j in range(1, m + 1)]
    z = np.zeros(n); N = np.zeros((n, n))
    for j in range(1, m + 2):
        d = gaps[j - 1]
        if d == 0.0:
            continue
        for i in range(n):
            for k in range(n):
                if i != k and Sm[i, k] == 0.0:
                    continue
                I = alpha[j - 1] @ _vanloan(Sm, i, k, d) @ beta[j] / Z
                if i == k:
                    z[i] += I
                else:
                    N[i, k] += I * Sm[i, k]
    p = alpha[m + 1] / Z                             # weights of the state at y, before the terminal factor
    if kind == "exact":
        ex = p * s
    elif kind == "right":
        zz, NN, ex = _full(Sm, s, p); z += zz; N += NN
    else:
        full = _full(Sm, s, p)
        tail = tu._num(Sm, s, p, u - y)
        z += full[0] - tail[0]; N += full[1] - tail[1]; ex = full[2] - tail[2]
    return z, N, ex, pi * beta[0] / Z, xs


def _draw(R, s, y, kind, vt, vm, u=None, pi=None, count=DRAWS, seed=0x9A1):
    Sm = tu._S(R, s); n = s.shape[0]; m = len(vt)
    off = np.arange(count + 1, dtype=np.int64) * m
    B, N, z, X, err = pp.panel_paths(seed, 3, np.full(count, y), np.full(count, 0 if kind == "exact" else 1),
                                     off, np.tile(vt, count), np.tile(np.asarray(vm, dtype=np.uint32), count),
                                     Sm.ravel(order="F"), s, u=None if u is None else np.full(count, u), pi=pi, states=True)
    assert err == 0
    return Sm, B, N.reshape(count, n, n, order="F"), z, X.reshape(count, m)


def _close(samples, exact, what, k=5.0):
    """Sample mean within k standard errors (plus a rounding floor) of the exact value, entry by entry."""
    samples = np.asarray(samples, dtype=float)
    mean = samples.mean(0); se = samples.std(0) / np.sqrt(samples.shape[0])
    bad = np.abs(mean - exact) > k * se + 1e-9
    assert not bad.any(), (what, np.argwhere(bad)[:5], mean[bad][:5], np.asarray(exact)[bad][:5], se[bad][:5])


def _check_law(R, s, y, kind, vt, vm, u=None, pi=None):
    n = s.shape[0]
    Sm, B, N, z, X = _draw(R, s, y, kind, vt, vm, u=u, pi=pi)
    pe = np.eye(n)[0] if pi is None else np.asarray(pi, dtype=float)
    ez, eN, eex, ea, exs = panel_expectations(Sm, s, pe, y, kind, vt, vm, u=u)
    _close(z, ez, "sojourn")
    off = ~np.eye(n, dtype=bool)
    _close(N[:, off], eN[off], "transitions")
    _close(N[:, np.arange(n), np.arange(n)], eex, "exits")
    _close(np.eye(n)[B], ea, "start state")
    for j in range(len(vt)):
        assert all((vm[j] >> c) & 1 for c in np.unique(X[:, j]))
        _close(np.eye(n)[X[:, j]], exs[j], "visit %d" % j)


CASES = {
    # the tied Coxian observed in its two stages at enrolment (t = 0) and twice after, exact absorption
    "tied_coxian_stages": (tu._tied_coxian(), 2.0, "exact", [0.0, 0.7, 1.5], [STAGES_COX[0], STAGES_COX[0], STAGES_COX[1]], None, None),
    # the complex R4 with a general pi, interval-censored terminal and a visit at t = y
    "r4_interval_visit_at_y": ((tu.R4, tu.S4), 1.0, "interval", [0.2, 0.6, 1.0], [0b0011, 0b0100, 0b1100], 1.8,
                               np.array([0.4, 0.3, 0.2, 0.1])),
    # general pi, exact at y with the phase seen at y and at enrolment
    "r4_exact_t0_ty": ((tu.R4, tu.S4), 1.2, "exact", [0.0, 0.5, 1.2], [0b0110, 0b1001, 0b1000], None, np.array([0.1, 0.5, 0.2, 0.2])),
    # right-censored, stage masks, general pi
    "r4_right": ((tu.R4, tu.S4), 1.5, "right", [0.4, 1.1], [0b0101, 0b1010], None, np.array([0.25, 0.25, 0.25, 0.25])),
    # a failure before the first inspection (y = 0, u > 0) with the stage seen at t = 0
    "r4_left_censored": ((tu.R4, tu.S4), 0.0, "interval", [0.0], [0b0011], 0.9, np.array([0.3, 0.3, 0.2, 0.2])),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_law_against_exact_values(name):
    (R, s), y, kind, vt, vm, u, pi = CASES[name]
    _check_law(R, s, y, kind, vt, vm, u=u, pi=pi)


def test_law_dense8_singletons():
    """Dense n = 8 with singleton masks taken from a path of the chain (so the data are possible), right-censored."""
    R, s = util.dense_rates(8, np.random.default_rng(8))
    vt, vm = [0.3, 0.9], [1 << 3, 1 << 6]
    _check_law(R, s, 1.4, "right", vt, vm)


def test_all_phase_masks_give_the_law_without_visits():
    """A mask of every phase carries nothing beyond "alive at t": the law is that of the observation without visits."""
    R, s = tu.R4, tu.S4
    pi = np.array([0.4, 0.3, 0.2, 0.1])
    for kind, y, u in (("exact", 1.3, None), ("right", 1.3, None), ("interval", 0.8, 1.7)):
        Sm, B, N, z, X = _draw(R, s, y, kind, [0.2, 0.5, 0.8], [0b1111] * 3, u=u, pi=pi, count=DRAWS // 2)
        ez, eN, eex, ea = tu.expectations(Sm, s, pi, y, kind, u=u)
        _close(z, ez, kind + " sojourn")
        off = ~np.eye(4, dtype=bool)
        _close(N[:, off], eN[off], kind + " transitions")
        _close(np.eye(4)[B], ea, kind + " start state")


def test_singleton_masks_pass_through_the_phase():
    """On every draw the path is in the observed phase at every visit time: the drawn state is that phase, and the path
    spends time in it (the Coxian moves forward only, so it also entered each observed phase exactly once)."""
    R, s = tu._tied_coxian()
    vt, vm = [0.5, 1.0, 1.6], [1 << 1, 1 << 2, 1 << 2]
    Sm, B, N, z, X = _draw(R, s, 2.2, "right", vt, vm, count=20_000)
    assert (X == np.array([1, 2, 2])).all()
    assert (z[:, 1] > 0).all() and (z[:, 2] > 0).all()
    assert (N[:, 0, 1] == 1).all() and (N[:, 1, 2] == 1).all() and (B == 0).all()


def test_long_panel_does_not_underflow():
    """One observation with 1000 visits (stage masks, every 0.05 over [0.05, 50]): the data probability is far below the
    smallest double, and the rescaled backward pass still draws every path."""
    R = np.array([[0.0, 2.0, 0.0, 0.0], [1.0, 0.0, 2.0, 0.0], [0.0, 1.0, 0.0, 2.0], [0.0, 0.0, 1.0, 0.0]])
    s = np.array([0.0, 0.0, 0.0, 0.01])
    rng = np.random.default_rng(1000)
    vt = 0.05 * np.arange(1, 1001)
    vm = [STAGES_COX[int(b)] for b in rng.integers(0, 2, 1000)]
    Sm, B, N, z, X = _draw(R, s, 50.0, "right", list(vt), vm, count=16)
    assert np.isfinite(z).all() and (z.sum(1) >= 50.0 * (1 - 1e-12)).all()
    for j in range(1000):
        assert all((vm[j] >> int(c)) & 1 for c in X[:, j])
