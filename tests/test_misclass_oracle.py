"""Misclassified panel observations (method 64 with stage visits) in the host build of the sampler,
oracle/pht_oracle_misclass.c: the paths have the exact conditional law given the start distribution, the emission matrix,
the stage readings and the terminal information.  The exact values come from a forward-backward pass over the visits with
the emission columns in place of the mask indicators (scipy expm per gap) and the Van Loan integrals per gap; the
tolerances from the Monte Carlo standard errors of ~2e5 host draws."""
import numpy as np
import pytest
import scipy.linalg as sl

from oracle import pyoracle_misclass as pm
from oracle import pyoracle_panel as pp
from tests import test_panel_oracle as tp
from tests import test_unif_oracle as tu
from tests import util

DRAWS = 200_000

# the tied Coxian (4 phases, forward only) read in 3 stages: phases 0-1 stage 0, phase 2 stage 1, phase 3 stage 2, with
# misreadings into the adjacent stages
E_COX = np.array([[0.9, 0.1, 0.0],
                  [0.8, 0.2, 0.0],
                  [0.1, 0.8, 0.1],
                  [0.0, 0.15, 0.85]])
# the complex R4 read in 2 stages with misreadings both ways
E_R4 = np.array([[0.85, 0.15], [0.7, 0.3], [0.2, 0.8], [0.05, 0.95]])


def emis_expectations(Sm, s, pi, y, kind, vt, vo, E, u=None):
    """Exact E[z], E[N_ij] (i != j), E[exits], P(start = a) and P(x_j = c) of a path with stage readings vo through E."""
    n = s.shape[0]
    ind = [E[:, o] for o in vo]
    times = [0.0] + list(vt) + [y]
    gaps = np.diff(times)
    m = len(vt)
    if kind == "exact":
        v = s.copy()
    elif kind == "right":
        v = np.ones(n)
    else:
        v = 1.0 - sl.expm(Sm * (u - y)) @ np.ones(n)
    Eg = [sl.expm(Sm * g) for g in gaps]
    beta = [None] * (m + 2)
    beta[m + 1] = v
    for j in range(m, 0, -1):
        beta[j] = ind[j - 1] * (Eg[j] @ beta[j + 1])
    beta[0] = Eg[0] @ beta[1]
    alpha = [pi.astype(float)]
    for j in range(1, m + 1):
        alpha.append((alpha[j - 1] @ Eg[j - 1]) * ind[j - 1])
    alpha.append(alpha[m] @ Eg[m])
    Z = pi @ beta[0]
    xs = [alpha[j] * (Eg[j] @ beta[j + 1]) / Z for j in range(1, m + 1)]
    z = np.zeros(n); N = np.zeros((n, n))
    for j in range(1, m + 2):
        d = gaps[j - 1]
        if d == 0.0:
            continue
        for i in range(n):
            for k in range(n):
                if i != k and Sm[i, k] == 0.0:
                    continue
                I = alpha[j - 1] @ tp._vanloan(Sm, i, k, d) @ beta[j] / Z
                if i == k:
                    z[i] += I
                else:
                    N[i, k] += I * Sm[i, k]
    p = alpha[m + 1] / Z
    if kind == "exact":
        ex = p * s
    elif kind == "right":
        zz, NN, ex = tp._full(Sm, s, p); z += zz; N += NN
    else:
        full = tp._full(Sm, s, p)
        tail = tu._num(Sm, s, p, u - y)
        z += full[0] - tail[0]; N += full[1] - tail[1]; ex = full[2] - tail[2]
    return z, N, ex, pi * beta[0] / Z, xs


def _draw(R, s, y, kind, vt, vo, E, u=None, pi=None, count=DRAWS, seed=0x3C1):
    Sm = tu._S(R, s); n = s.shape[0]; m = len(vt)
    off = np.arange(count + 1, dtype=np.int64) * m
    B, N, z, X, err = pm.misclass_paths(seed, 3, np.full(count, y), np.full(count, 0 if kind == "exact" else 1), off,
                                        np.tile(vt, count), np.tile(np.asarray(vo, dtype=np.uint32), count), E,
                                        Sm.ravel(order="F"), s, u=None if u is None else np.full(count, u), pi=pi, states=True)
    assert err == 0
    return Sm, B, N.reshape(count, n, n, order="F"), z, X.reshape(count, m)


def _check_law(R, s, y, kind, vt, vo, E, u=None, pi=None):
    n = s.shape[0]
    Sm, B, N, z, X = _draw(R, s, y, kind, vt, vo, E, u=u, pi=pi)
    pe = np.eye(n)[0] if pi is None else np.asarray(pi, dtype=float)
    ez, eN, eex, ea, exs = emis_expectations(Sm, s, pe, y, kind, vt, vo, E, u=u)
    tp._close(z, ez, "sojourn")
    off = ~np.eye(n, dtype=bool)
    tp._close(N[:, off], eN[off], "transitions")
    tp._close(N[:, np.arange(n), np.arange(n)], eex, "exits")
    tp._close(np.eye(n)[B], ea, "start state")
    for j in range(len(vt)):
        assert (E[np.unique(X[:, j]), vo[j]] > 0).all()
        tp._close(np.eye(n)[X[:, j]], exs[j], "visit %d" % j)


CASES = {
    # the tied Coxian read with off-diagonal misreadings at enrolment (t = 0) and three times after, exact absorption
    "tied_coxian_3stage": (tu._tied_coxian(), E_COX, 2.0, "exact", [0.0, 0.6, 1.2, 1.7], [0, 1, 1, 2], None, None),
    # a stage regression (stage 2 read, then stage 1): no forward-only path has it as masks, the emission form draws it
    "tied_coxian_regression": (tu._tied_coxian(), E_COX, 2.5, "right", [0.5, 1.4, 2.0], [0, 2, 1], None, None),
    # the complex R4 with a general pi, interval-censored terminal and a visit at t = y
    "r4_interval_visit_at_y": ((tu.R4, tu.S4), E_R4, 1.0, "interval", [0.2, 0.6, 1.0], [0, 1, 1], 1.8,
                               np.array([0.4, 0.3, 0.2, 0.1])),
    # general pi, exact at y with readings at enrolment and at y
    "r4_exact_t0_ty": ((tu.R4, tu.S4), E_R4, 1.2, "exact", [0.0, 0.5, 1.2], [1, 0, 1], None, np.array([0.1, 0.5, 0.2, 0.2])),
    # right-censored, general pi
    "r4_right": ((tu.R4, tu.S4), E_R4, 1.5, "right", [0.4, 1.1], [0, 1], None, np.array([0.25, 0.25, 0.25, 0.25])),
    # a failure before the first inspection (y = 0, u > 0) with the stage read at t = 0
    "r4_left_censored": ((tu.R4, tu.S4), E_R4, 0.0, "interval", [0.0], [1], 0.9, np.array([0.3, 0.3, 0.2, 0.2])),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_law_against_exact_values(name):
    (R, s), E, y, kind, vt, vo, u, pi = CASES[name]
    _check_law(R, s, y, kind, vt, vo, E, u=u, pi=pi)


def test_law_dense8():
    """Dense n = 8 read in 3 stages through a dense E (every phase can be read as every stage), right-censored."""
    rng = np.random.default_rng(8)
    R, s = util.dense_rates(8, rng)
    E = rng.dirichlet(np.ones(3), 8)
    _check_law(R, s, 1.4, "right", [0.3, 0.9], [2, 0], E)


def test_indicator_E_gives_the_mask_paths_bit_for_bit():
    """E the 0/1 indicator of the Coxian's two 2-phase stages: every path, statistic and visit state is the mask form's."""
    R, s = tu._tied_coxian()
    Sm = tu._S(R, s)
    E = np.array([[1.0, 0.0], [1.0, 0.0], [0.0, 1.0], [0.0, 1.0]])
    rng = np.random.default_rng(5)
    count = 4000
    y = rng.uniform(0.5, 3.0, count); cens = rng.integers(0, 2, count)
    m = rng.integers(0, 4, count)
    off = np.concatenate([[0], np.cumsum(m)]).astype(np.int64)
    t = np.concatenate([np.sort(rng.uniform(0, yk, mk)) for yk, mk in zip(y, m)])
    # stages along a forward path: never back from stage 1 to stage 0
    st = np.concatenate([np.sort(rng.integers(0, 2, mk)) for mk in m]).astype(np.uint32)
    masks = np.array([0b0011, 0b1100], dtype=np.uint32)[st]
    a = pm.misclass_paths(11, 2, y, cens, off, t, st, E, Sm.ravel(order="F"), s, states=True)
    b = pp.panel_paths(11, 2, y, cens, off, t, masks, Sm.ravel(order="F"), s, states=True)
    assert a[-1] == 0 and b[-1] == 0
    for x, w in zip(a[:-1], b[:-1]):
        assert np.array_equal(x, w)


def test_regression_is_refused_as_masks_and_drawn_as_stages():
    """The regression of "tied_coxian_regression" as stage masks has no path: the mask form finds only zero weights
    (error 512), the emission form draws every path."""
    R, s = tu._tied_coxian()
    Sm = tu._S(R, s)
    vt, vo = [0.5, 1.4, 2.0], [0, 2, 1]
    cols = np.array([1 << 0 | 1 << 1, 1 << 2, 1 << 3], dtype=np.uint32)
    off = np.array([0, 3], dtype=np.int64)
    *_, err = pp.panel_paths(1, 1, [2.5], [1], off, vt, cols[vo], Sm.ravel(order="F"), s)
    assert err == 512
    *_, X, err = pm.misclass_paths(1, 1, [2.5], [1], off, vt, np.array(vo, dtype=np.uint32), E_COX, Sm.ravel(order="F"), s,
                                   states=True)
    assert err == 0 and (np.diff(X) >= 0).all() and (E_COX[X, vo] > 0).all()
