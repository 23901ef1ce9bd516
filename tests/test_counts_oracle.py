"""Records with counts (method 64, Engine.set_counts) in the sampler's host build: the record form of pht_unif.h (one
preparation per record, then its units) draws every unit's path bit for bit as pht_unif_path draws the matching
observation of the expanded data np.repeat(records, counts); and synth.tabulate round-trips through np.repeat."""
import numpy as np
import pytest

from oracle import pyoracle_counts as pc
from oracle import pyoracle_unif as pu
from phasetype_b200 import synth
from tests.test_unif_oracle import GENERATORS, _S


def _records(rng, l, n, cens_mix=True):
    """l records: exact, right-, interval- and left-censored (y = 0 with a finite u), counts 0 .. 40."""
    kind = rng.integers(0, 4 if cens_mix else 1, l)
    y = rng.uniform(0.05, 2.5, l)
    cens = (kind > 0).astype(np.int32)
    u = np.full(l, np.inf)
    iv = kind >= 2
    u[iv] = y[iv] + rng.uniform(0.1, 1.5, iv.sum())
    y[kind == 3] = 0.0
    counts = rng.integers(0, 41, l).astype(np.uint32)
    counts[0] = 0
    return y, cens, u, counts


def _compare(Sm, s, y, cens, u, counts, pi, kb, seed=11, it=3):
    B, N, z, err = pc.record_paths(seed, it, y, cens, counts, Sm.ravel(order="F"), s, u=u, pi=pi, kb=kb)
    Be, Ne, ze, erre = pu.unif_paths(seed, it, np.repeat(y, counts), np.repeat(cens, counts), Sm.ravel(order="F"), s,
                                     u=np.repeat(u, counts), pi=pi)
    assert err == erre == 0
    assert B.shape == Be.shape and np.array_equal(B, Be)
    assert np.array_equal(N, Ne)
    assert np.array_equal(z.view(np.uint64), ze.view(np.uint64))
    return B.shape[0]


@pytest.mark.parametrize("name", ["erlang4", "complex_r4", "dense32", "stiff", "sm"])
@pytest.mark.parametrize("general_pi", [False, True])
def test_record_form_equals_per_observation_paths(name, general_pi):
    R, s = GENERATORS[name]
    Sm = _S(R, s); n = s.shape[0]
    rng = np.random.default_rng(hash((name, general_pi)) & 0xffff)
    y, cens, u, counts = _records(rng, 24 if n < 32 else 8, n)
    if name == "stiff":                       # lambda ~ 1000: K(lambda y) near the table's cap of 4096 powers
        y = np.minimum(y, 1.0); u = np.where(np.isfinite(u), np.minimum(u, y + 2.0), u)
    pi = rng.dirichlet(np.ones(n)) if general_pi else None
    assert _compare(Sm, s, y, cens, u, counts, pi, kb=255) > 0


@pytest.mark.parametrize("kb", [0, 3, 17])
def test_weights_beyond_the_buffer_are_recomputed(kb):
    """K(lambda y) far above the buffer bound: the weights past kb come from pht_unif_w, with the same bits."""
    R, s = GENERATORS["complex_r4"]
    Sm = _S(R, s); n = s.shape[0]
    rng = np.random.default_rng(kb)
    y, cens, u, counts = _records(rng, 20, n)
    _compare(Sm, s, y, cens, u, counts, rng.dirichlet(np.ones(n)), kb=kb)


def test_all_ones_and_zero_counts():
    R, s = GENERATORS["erlang4"]
    Sm = _S(R, s)
    rng = np.random.default_rng(4)
    y, cens, u, _ = _records(rng, 30, 4)
    assert _compare(Sm, s, y, cens, u, np.ones(30, dtype=np.uint32), None, kb=255) == 30
    B, N, z, err = pc.record_paths(1, 1, y, cens, np.zeros(30, dtype=np.uint32), Sm.ravel(order="F"), s, u=u)
    assert err == 0 and B.shape == (0,)


def test_tabulate_round_trips():
    rng = np.random.default_rng(9)
    R, s = GENERATORS["erlang4"]
    y, u, cens, _ = synth.inspection(R, s, 5000, 0.25, 12, rng)
    ty, tc, tu, w = synth.tabulate(y, cens, u)
    assert ty.shape[0] <= 13 and int(w.sum()) == 5000 and w.dtype == np.uint32
    # first-occurrence order, and the expansion holds every observation as often as the data do
    first = [int(np.flatnonzero((y == a) & (u == b))[0]) for a, b in zip(ty, tu)]
    assert first == sorted(first)
    ey, ec, eu = np.repeat(ty, w), np.repeat(tc, w), np.repeat(tu, w)
    key = lambda a, c, b: sorted(zip(a.tolist(), c.tolist(), b.tolist()))
    assert key(ey, ec, eu) == key(y, cens, u)
    # without u, and with exact ties in y only
    yr = np.round(rng.exponential(1.0, 3000), 2); cr = (rng.random(3000) < 0.3).astype(np.int32)
    ty, tc, tu, w = synth.tabulate(yr, cr)
    assert tu is None and int(w.sum()) == 3000
    assert sorted(zip(np.repeat(ty, w).tolist(), np.repeat(tc, w).tolist())) == sorted(zip(yr.tolist(), cr.tolist()))
