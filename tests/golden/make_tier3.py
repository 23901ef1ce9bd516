"""Tier-3 fixture: the chain of the UNMODIFIED reference LJMA_Gibbs (oracle/_ref, built from $PHT_REFERENCE_SRC/src) on the
structured repairable-system model of the reference's tests/phtMCMC2.R with 400 simulated observations, for each of the
three methods.  Run with an upstream PhaseType source tree:  PHT_REFERENCE_SRC=<checkout> python tests/golden/make_tier3.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po          # noqa: E402
from tests import util                     # noqa: E402

po.build()
assert po.have_ref(), "the reference build (oracle/_ref) is needed"
rng = np.random.default_rng(8)
F, Rr = 1.5, 11.0
R = np.array([[0, F, F], [Rr, 0, 0], [Rr, 0, 0]], dtype=float); s = np.array([0.0, F, F])
y = util.simulate_pht(R, s, 400, rng); cens = np.zeros(400, dtype=np.int32)
T = np.array([0, 2, 2, 0, 1, 0, 0, 0, 1, 0, 0, 0, 0, 1, 1, 0], dtype=np.int32); Cm = np.ones(16)
nu = np.array([24.0, 180.0]); zeta = np.array([16.0, 16.0])
it = 1500
out = {"y": y, "cens": cens, "T": T, "C": Cm, "nu": nu, "zeta": zeta, "it": it}
for method in (1, 2, 4):
    out["chain_%d" % method] = po.ref_gibbs(5, False, it, 1, method, 3, nu, zeta, T, Cm, y, cens, [-1.0])
np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "chains", "tier3_reference_chain.npz"), **out)
print("written", {k: np.asarray(v).shape for k, v in out.items()})
