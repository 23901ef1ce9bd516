"""split_rhat (phasetype_b200/diagnostics.py) on the CPU: a case worked by hand, and its behaviour on chains that agree
and on chains that do not."""
import numpy as np
import pytest

from phasetype_b200.diagnostics import split_rhat


def test_hand_computed_case():
    # halves [1, 2], [3, 4], [2, 3], [4, 5]: W = 0.5, half means 1.5, 3.5, 2.5, 4.5 with variance 5/3, h = 2
    draws = np.array([[1.0, 2.0, 3.0, 4.0], [2.0, 3.0, 4.0, 5.0]])
    want = np.sqrt((0.5 * 0.5 + 5.0 / 3.0) / 0.5)
    assert split_rhat(draws) == pytest.approx(want, rel=1e-14)
    # (chains, sweeps, m) gives one value per parameter; an odd sweep count drops the middle draw
    both = np.stack([draws, 2.0 * draws], axis=2)
    assert np.allclose(split_rhat(both), [want, want], rtol=1e-14)
    odd = np.array([[1.0, 2.0, 99.0, 3.0, 4.0], [2.0, 3.0, -99.0, 4.0, 5.0]])
    assert split_rhat(odd) == pytest.approx(want, rel=1e-14)


def test_iid_chains_give_one_and_shifted_chains_do_not():
    rng = np.random.default_rng(5)
    iid = rng.normal(size=(8, 4000, 3))
    assert np.all(np.abs(split_rhat(iid) - 1.0) < 0.01)
    shifted = iid + np.arange(8)[:, None, None] * 0.5
    assert np.all(split_rhat(shifted) > 1.5)
    # a trend inside every chain shows between the halves even when the chains agree with each other
    trend = iid + np.linspace(0.0, 3.0, 4000)[None, :, None]
    assert np.all(split_rhat(trend) > 1.2)


def test_too_few_draws_refused():
    with pytest.raises(ValueError):
        split_rhat(np.zeros((4, 3, 2)))
