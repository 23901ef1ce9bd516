"""The CPU restatement of the interval-censored MHRS sampler (oracle pho_mhrs_paths_iv) on its own: with every bound
+inf it is the right-censored sampler bit for bit, and its rejection loop needs 1 / P(y <= T <= u) attempts per path."""
import numpy as np
import scipy.linalg as sl

from oracle import pyoracle as po
from oracle import pyoracle_iv as poi
from phasetype_b200 import synth
from tests import util


def _S(R, s):
    S = R.copy()
    np.fill_diagonal(S, -(R.sum(1) + s))
    return S


def test_infinite_bounds_are_the_right_censored_sampler():
    rng = np.random.default_rng(17)
    R, s = util.dense_rates(6, rng)
    S = _S(R, s).ravel(order="F").copy()
    y = rng.exponential(1.2, 2000) + 0.01
    cens = (rng.uniform(size=2000) < 0.5).astype(np.int32)
    for mhit in (1, 3):
        a = po.mhrs_paths("oracle", 21, 4, y, cens, S, s, mhit=mhit)
        b = poi.mhrs_paths_iv(21, 4, y, cens, np.full(2000, np.inf), S, s, mhit=mhit)
        for x, z in zip(a[:3], b[:3]):
            assert np.array_equal(x, z)
        assert a[3] == b[3]


def test_attempts_per_path_follow_the_interval_probability():
    rng = np.random.default_rng(23)
    R, s = util.dense_rates(4, rng)
    S = _S(R, s)
    l = 20000
    for y0, u0 in ((0.5, 0.8), (2.0, 2.1), (0.1, 4.0)):
        y = np.full(l, y0); u = np.full(l, u0); cens = np.ones(l, dtype=np.int32)
        _, _, z, cnt = poi.mhrs_paths_iv(5, 1, y, cens, u, S.ravel(order="F").copy(), s)
        surv = lambda t: sl.expm(S * t)[0].sum()          # P(T > t), start in state 0
        p = surv(y0) - surv(u0)
        mean = cnt["attempts"] / l
        sd = np.sqrt((1 - p) / p ** 2 / l)                # the attempt count per path is Geometric(p)
        assert abs(mean - 1 / p) < 5 * sd, (y0, u0, mean, 1 / p, sd)
        t = z.sum(1)
        assert (t >= y0 * (1 - 1e-12)).all() and (t <= u0 * (1 + 1e-12)).all()


def test_inspection_generator():
    R, s = util.coxian_rates(4)
    y, u, cens, t = synth.inspection(R, s, 5000, 0.7, 6, np.random.default_rng(3))
    iv = np.isfinite(u)
    assert (cens == 1).all() and (y > 0).all()
    assert (y[iv] < t[iv]).all() and (t[iv] <= u[iv]).all() and np.allclose(u[iv] - np.where(y[iv] > 1e-9, y[iv], 0), 0.7)
    assert (t[~iv] > 6 * 0.7).all() and (y[~iv] == 6 * 0.7).all()
