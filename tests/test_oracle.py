"""The CPU restatement (oracle/pht_oracle.c) against (1) the committed golden vectors dumped from the
unmodified reference C, (2) the reference build itself where PHT_REFERENCE_SRC names its sources, (3) the analytic
Hobolth-Jensen conditional expectations (tier 2), (4) the reference's whole LJMA_Gibbs (tier 3)."""
import glob
import os

import numpy as np
import pytest
import scipy.linalg as sl

from oracle import pyoracle as po
from phasetype_b200 import synth
from tests import util

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz")))
needs_ref = pytest.mark.skipif(not po.have_ref(), reason="oracle/_ref (reference build) not present")


def golden_run(impl, g):
    if str(g["method"]) == "MHRS":
        return po.mhrs_paths(impl, int(g["seed"]), int(g["it"]), g["y"], g["cens"], g["S"], g["s"], mhit=int(g["mhit"]))
    return po.spectral_paths(impl, str(g["method"]), int(g["seed"]), int(g["it"]), g["y"], g["cens"], g["S"], g["s"],
                             spectral=(g["evals"], g["Q"], g["Qinv"]))


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_oracle_reproduces_golden_vectors(path):
    g = np.load(path)
    B, N, z, _ = golden_run("oracle", g)
    assert np.array_equal(B, g["B"]) and np.array_equal(N, g["N"]) and np.array_equal(z, g["z"])


@needs_ref
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_reference_build_reproduces_golden_vectors(path):
    g = np.load(path)
    B, N, z, _ = golden_run("ref", g)
    assert np.array_equal(B, g["B"]) and np.array_equal(N, g["N"]) and np.array_equal(z, g["z"])


def _S(R, s):
    n = s.shape[0]; S = R.copy()
    for i in range(n):
        S[i, i] = -(R[i].sum() + s[i])
    return S.ravel(order="F").copy()


@needs_ref
@pytest.mark.parametrize("method,n,kind,fc", [("MHRS", 3, "dense", 0.3), ("MHRS", 16, "dense", 0.2), ("MHRS", 32, "dense", 0.0),
                                              ("DCS", 16, "sym", 0.0), ("DCS", 32, "sym", 0.0), ("ECS", 8, "sym", 0.5),
                                              ("ECS", 32, "sym", 0.2), ("ECS", 6, "coxian", 0.2), ("DCS", 6, "coxian", 0.0)])
def test_oracle_equals_reference_bit_for_bit(method, n, kind, fc):
    rng = np.random.default_rng(n * 7 + len(method))
    R, s = util.coxian_rates(n) if kind == "coxian" else util.dense_rates(n, rng, symmetric=(kind == "sym"))
    S = _S(R, s)
    l = 600 if n <= 16 else 150
    y = rng.exponential(1.2, l) + 0.01; cens = (rng.uniform(size=l) < fc).astype(np.int32)
    if method == "MHRS":
        a = po.mhrs_paths("oracle", 5, 2, y, cens, S, s, mhit=2); b = po.mhrs_paths("ref", 5, 2, y, cens, S, s, mhit=2)
        assert a[3]["attempts"] == b[3]["attempts"] and a[3]["jumps"] == b[3]["jumps"]
    else:
        spec = po.eigen("ref", S, n)
        a = po.spectral_paths("oracle", method, 5, 2, y, cens, S, s, spectral=spec)
        b = po.spectral_paths("ref", method, 5, 2, y, cens, S, s, spectral=spec)
    for u, v in zip(a[:3], b[:3]):
        assert np.array_equal(u, v)


@needs_ref
@pytest.mark.parametrize("variant", ["MHS_HOBOLTH", "MHS_ASLETT"])
@pytest.mark.parametrize("n,zero_exits,mhit", [(3, False, 1), (5, True, 3), (8, False, 0), (16, False, 2)])
def test_dead_variants_equal_reference_bit_for_bit(variant, n, zero_exits, mhit):
    """SURVEY 8(f)1: LJMA_MHsample_Hobolth / LJMA_MHsample_Aslett have no caller in the reference, but they are external
    symbols of its build; the restatement is pinned against them, chain = sub-stream (every chain ends with LJMA_GUI())."""
    rng = np.random.default_rng(31 * n + mhit)
    R, s = util.dense_rates(n, rng, symmetric=True)
    if zero_exits:
        s[1] = 0.0; s[3] = 0.0            # states that cannot exit: the retry loops run
    S = _S(R, s)
    l = 400 if n <= 8 else 120
    y = util.simulate_pht(R, s, l, rng); cens = (rng.uniform(size=l) < 0.25).astype(np.int32)
    spec = po.eigen("ref", S, n)
    a = po.mh_variant_paths("oracle", variant, 5, 2, y, cens, S, s, mhit=mhit, spectral=spec)
    b = po.mh_variant_paths("ref", variant, 5, 2, y, cens, S, s, mhit=mhit, spectral=spec)
    for u, v in zip(a[:3], b[:3]):
        assert np.array_equal(u, v)


@pytest.mark.parametrize("variant", ["MHS_HOBOLTH", "MHS_ASLETT"])
def test_dead_variants_reach_the_conditional_law(variant):
    """Tier 2 for the MH variants: with enough MH proposals the chain statistics match the analytic conditional
    expectations given absorption AT y (Hobolth-Jensen), although the chain samplers only condition on `alive at y`."""
    Sm = np.array([[-4.1, 1.8, 1.8], [9.5, -11.3, 0.0], [9.5, 0.0, -15.5]]); s = -Sm.sum(1)
    y0, l = 1.5, 20000
    y = np.full(l, y0); cens = np.zeros(l, dtype=np.int32)
    B, N, z, _ = po.mh_variant_paths("oracle", variant, 42, 1, y, cens, Sm.ravel(order="F").copy(), s, mhit=25)
    Ez, EN, exit_p = hobolth_jensen(Sm, s, y0, False)
    Nm = N.mean(0).reshape(3, 3, order="F")
    assert np.abs(z.mean(0) - Ez).max() < 5 * z.std(0).max() / np.sqrt(l) + 2e-3
    off = ~np.eye(3, dtype=bool)
    assert np.abs(Nm[off] - EN[off]).max() < 0.04
    assert np.abs(np.diag(Nm) - exit_p).max() < 0.015


@needs_ref
def test_lapack_binding_matches_reference_eigen():
    rng = np.random.default_rng(0)
    R, s = util.dense_rates(8, rng, symmetric=True)
    S = _S(R, s)
    for u, v in zip(po.eigen("oracle", S, 8), po.eigen("ref", S, 8)):
        assert np.array_equal(u, v)


def test_native_spectral_solver_invariants():
    """pht_eigen.h (the engine's solver) against LAPACK/expm through quantities that do not depend on eigenvalue
    order or eigenvector scaling."""
    for n, kind in [(1, "sym"), (2, "sym"), (3, "sym"), (8, "sym"), (16, "sym"), (32, "sym"), (4, "coxian"), (8, "coxian")]:
        for trial in range(5):
            rng = np.random.default_rng(100 * n + trial)
            R, s = util.coxian_rates(n) if kind == "coxian" else util.dense_rates(n, rng, symmetric=True)
            S = _S(R, s); Sm = S.reshape(n, n, order="F")
            ev, Q, Qi = po.eigen("native", S, n)
            Qm = Q.reshape(n, n, order="F"); Qim = Qi.reshape(n, n, order="F")
            tol = 1e-13 * max(1.0, np.linalg.cond(Qm))
            assert np.abs(Qm @ np.diag(ev) @ Qim - Sm).max() <= tol * np.abs(Sm).max()
            assert np.abs(Qm @ Qim - np.eye(n)).max() <= tol
            assert np.abs(np.sort(ev) - np.sort(np.linalg.eigvals(Sm).real)).max() <= tol * np.abs(ev).max()
            assert np.abs(Qm @ np.diag(np.exp(1.3 * ev)) @ Qim - sl.expm(1.3 * Sm)).max() <= 10 * tol
            assert np.allclose(np.linalg.norm(Qm, axis=0), 1.0)
    R, s = util.dense_rates(8, np.random.default_rng(5))          # unsymmetric dense: complex pairs, must be flagged
    with pytest.raises(ValueError):
        po.eigen("native", _S(R, s), 8)


# ---------------------------------------------------------------- tier 2: analytic conditional expectations
def hobolth_jensen(Sm, s, y, censored):
    """E[z_i | y], E[N_ij | y], exit-state probabilities for pi = e1 (SURVEY.md section 8(c); Van Loan block integrals)."""
    n = s.shape[0]
    pi = np.zeros(n); pi[0] = 1.0
    v = np.ones(n) if censored else s
    a = pi @ sl.expm(Sm * y)
    f = a @ v
    Ez = np.zeros(n); EN = np.zeros((n, n))
    for i in range(n):
        for j in range(n):
            E = np.zeros((n, n)); E[i, j] = 1.0
            A = np.block([[Sm, E], [np.zeros((n, n)), Sm]])
            I = sl.expm(A * y)[:n, n:]            # int_0^y e^{Su} E e^{S(y-u)} du
            val = pi @ I @ v / f
            if i == j:
                Ez[i] = val
            else:
                EN[i, j] = Sm[i, j] * val
    if censored:
        post = a @ np.linalg.inv(-Sm) / f         # expected time per state after y until absorption
        Ez = Ez + post
        EN = EN + (post[:, None] * Sm) * (1 - np.eye(n))
        exit_p = post * s
    else:
        exit_p = a * s / f
    return Ez, EN, exit_p


@pytest.mark.parametrize("method,censored", [("ECS", False), ("DCS", False), ("ECS", True), ("MHRS", True)])
def test_conditional_expectations_match_hobolth_jensen(method, censored):
    Sm = np.array([[-4.1, 1.8, 1.8], [9.5, -11.3, 0.0], [9.5, 0.0, -15.5]]); s = -Sm.sum(1)       # SURVEY 8(c), unequal exits
    y0, l = 1.5, 40000
    y = np.full(l, y0); cens = np.full(l, 1 if censored else 0, dtype=np.int32)
    S = Sm.ravel(order="F").copy()
    if method == "MHRS":
        B, N, z, _ = po.mhrs_paths("oracle", 42, 1, y, cens, S, s, mhit=0)
    else:
        B, N, z, _ = po.spectral_paths("oracle", method, 42, 1, y, cens, S, s)
    Ez, EN, exit_p = hobolth_jensen(Sm, s, y0, censored)
    Nm = N.mean(0).reshape(3, 3, order="F")
    assert np.abs(z.mean(0) - Ez).max() < 4 * z.std(0).max() / np.sqrt(l) + 1e-3
    off = ~np.eye(3, dtype=bool)
    assert np.abs(Nm[off] - EN[off]).max() < 0.03
    assert np.abs(np.diag(Nm) - exit_p).max() < 0.012
    if not censored:
        assert np.allclose(exit_p, [0.3171, 0.2036, 0.4793], atol=2e-4)          # known answer quoted in SURVEY.md
        assert np.allclose(Ez, [1.18422, 0.19245, 0.12333], atol=2e-5)


# ---------------------------------------------------------------- tier 3 and driver parity against the reference's LJMA_Gibbs
@needs_ref
def test_driver_matches_reference_gibbs_on_one_phase_model():
    """n = 1: the spectral data are trivially identical (Q = 1), so the reference's own LJMA_Gibbs, driven through the
    keyed stream hook, and the restated driver differ only in how z is summed (double vs fixed point)."""
    rng = np.random.default_rng(3)
    y = rng.exponential(0.7, 500) + 0.01; cens = np.zeros(500, dtype=np.int32)
    T = np.array([0, 0, 1, 0], dtype=np.int32); Cm = np.ones(4)
    for method in (2, 4):
        a, _ = po.gibbs(77, 40, 1, method, 1, [2.0], [1.5], T, Cm, y, cens, [-1.0])
        b = po.ref_gibbs(77, True, 40, 1, method, 1, [2.0], [1.5], T, Cm, y, cens, [-1.0])
        assert np.allclose(a, b, rtol=1e-12, atol=0)


@needs_ref
@pytest.mark.parametrize("method", [1, 2, 4])
def test_posterior_agrees_with_reference_chain(method):
    """Structured repairable-system model of tests/phtMCMC2.R (identifiable: 2 parameters) on 400 simulated
    observations: posterior means of the restated chain and of the reference's LJMA_Gibbs agree within Monte-Carlo error."""
    rng = np.random.default_rng(8)
    F, Rr = 1.5, 11.0
    R = np.array([[0, F, F], [Rr, 0, 0], [Rr, 0, 0]], dtype=float); s = np.array([0.0, F, F])
    y = util.simulate_pht(R, s, 400, rng); cens = np.zeros(400, dtype=np.int32)
    T = [0, 2, 2, 0, 1, 0, 0, 0, 1, 0, 0, 0, 0, 1, 1, 0]; Cm = np.ones(16)
    nu = [24.0, 180.0]; zeta = [16.0, 16.0]
    it = 1500
    a, _ = po.gibbs(5, it, 1, method, 3, nu, zeta, T, Cm, y, cens, [-1.0])
    b = po.ref_gibbs(5, False, it, 1, method, 3, nu, zeta, T, Cm, y, cens, [-1.0])
    for v in range(2):
        xa, xb = a[200:, v], b[200:, v]
        se = np.sqrt(xa.var() / 100 + xb.var() / 100)        # ~100 effective draws each (conservative)
        assert abs(xa.mean() - xb.mean()) < 4 * se
        assert abs(np.quantile(xa, 0.9) - np.quantile(xb, 0.9)) < 8 * se


def test_sharded_statistics_sum_to_the_whole():
    wl = synth.config(3, "MHRS", l=3000)
    zb = po.choose_zbits(wl.y.sum())
    whole = po.sweep_stats(9, 1, True, 1, 1, wl.n, wl.T, wl.C, wl.theta, wl.y, wl.censored, zbits=zb)
    parts = [po.sweep_stats(9, 1, True, 1, 1, wl.n, wl.T, wl.C, wl.theta, wl.y, wl.censored, rank=r, world=4, zbits=zb) for r in range(4)]
    for k in range(3):
        assert np.array_equal(whole[k], sum(p[k] for p in parts))


@pytest.mark.skipif(not po.have_ref_libm(), reason="oracle/_ref/libphtref_libm.so (make ref-libm) not present")
def test_libm_mismatch_rate_is_reported(tmp_path):
    """SURVEY H3: tier 1 is decided against the reference built with the engine's exp/log, plain-loop BLAS and
    -ffp-contract=off (`make ref`).  This test REPORTS what those three substitutions hide: the same reference sources
    with the platform's libm, OpenBLAS dgemv/dgemm and R's default -O2 (`make ref-libm`), run on the golden inputs
    and on a larger sample per method.  Where B and N agree the z totals must agree to 1e-12 relative for MHRS (north_star's
    tolerance; for the equation-solving samplers the figure is reported per component and bounded at 1e-12 of the path length); the rate at which an integer statistic differs (a flipped comparison somewhere on the path) is
    written to libm_mismatch.json in the test's temporary directory and printed (profiles/r2_libm_mismatch.json is a
    recorded copy), not asserted to be zero."""
    import json
    report = {}
    worst_z = 0.0; worst_path = 0.0
    cases = [(os.path.basename(p)[:-4], np.load(p)) for p in GOLDEN]
    rng = np.random.default_rng(2026)
    for method, n, kind, fc, l in (("MHRS", 8, "dense", 0.2, 20000), ("ECS", 8, "sym", 0.2, 4000), ("DCS", 8, "sym", 0.0, 4000)):
        R, s = util.dense_rates(n, rng, symmetric=(kind == "sym"))
        S = _S(R, s)
        g = dict(method=method, seed=77, it=2, mhit=1, y=rng.exponential(1.2, l) + 0.01, S=S, s=s)
        g["cens"] = (rng.uniform(size=l) < fc).astype(np.int32)
        if method != "MHRS":
            g["evals"], g["Q"], g["Qinv"] = po.eigen("ref", S, n)
        cases.append(("%s_n%d_l%d" % (method.lower(), n, l), g))
    for name, g in cases:
        B0, N0, z0, _ = golden_run("ref", g)
        B1, N1, z1, _ = golden_run("ref_libm", g)
        same = (B0 == B1) & (N0 == N1).all(1)
        rel = np.abs(z1[same] - z0[same]) / np.maximum(np.abs(z0[same]), 1e-300)
        rel = rel[z0[same] != 0.0]
        mz = float(rel.max()) if rel.size else 0.0
        # the same differences against the length of the path they belong to (a sojourn drawn by ARMS or Brent is
        # the solution of an equation in exp/log values: its own relative error is the solver's conditioning times
        # the libm difference, and a short sojourn shows it largest)
        tot = np.abs(z0[same]).sum(1, keepdims=True)
        mp_ = float((np.abs(z1[same] - z0[same]) / np.maximum(tot, 1e-300)).max()) if same.any() else 0.0
        if str(g["method"]) == "MHRS":
            worst_z = max(worst_z, mz)
        worst_path = max(worst_path, mp_)
        report[name] = {"paths": int(B0.shape[0]), "paths_with_different_B_or_N": int((~same).sum()),
                        "mismatch_rate": float((~same).mean()), "max_rel_z_error_where_B_N_agree": mz,
                        "max_z_error_relative_to_path_length": mp_}
    with open(tmp_path / "libm_mismatch.json", "w") as f:
        json.dump({"what": "reference C built with platform libm + OpenBLAS + default -O2 (make ref-libm) versus the tier-1 "
                           "checker build (make ref: pht_math.h exp/log, plain-loop BLAS, -ffp-contract=off), same Philox uniforms",
                   "cases": report}, f, indent=1, sort_keys=True)
    print("report:", tmp_path / "libm_mismatch.json")
    print(json.dumps(report, indent=1))
    # MHRS sojourns are sums of scale * (-log u): 1e-12 holds per component.  ECS / DCS sojourns are roots of equations
    # in exp/log values (ARMS inversion, Brent): per component they agree to ~1e-10, and to 1e-12 of the path length.
    assert worst_z <= 1e-12
    assert worst_path <= 1e-12
