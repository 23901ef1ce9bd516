"""Generate the golden vectors in this directory from the UNMODIFIED reference C (oracle/_ref, i.e.
$PHT_REFERENCE_SRC/src compiled against the R stand-in).  Run once with an upstream PhaseType source tree:

    PHT_REFERENCE_SRC=<PhaseType checkout> python tests/golden/make_golden.py

Each .npz holds the inputs (S, s, y, censored, seed, iteration, mhit, and for ECS/DCS the LAPACK spectral data
the reference itself computed) and the reference's per-observation outputs (B, N, z).  The reference's own
tests pin no numbers (SURVEY.md section 4), so these dumps are the pins."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po          # noqa: E402
from tests import util                     # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
Y20 = [1.45353415045187, 1.85349532001349, 2.01084961814576, 0.505725921290172, 1.56252630012213,
       3.41158665930278, 1.52674487509487, 4.3428662377235, 8.03208018151311, 2.41746547476986,
       0.38828086509283, 2.61513815012196, 3.39148865480856, 1.82705817807965, 1.42090953713845,
       0.851438991331866, 0.0178808867191894, 0.632198596390046, 0.959910259815998, 1.83344199966323]


def model(kind, n, rng):
    if kind == "package":        # man/PhaseType-package.Rd:39
        S = np.array([[-3.6, 1.8, 1.8], [9.5, -11.3, 0.0], [9.5, 0.0, -11.3]])
        R = S.copy(); np.fill_diagonal(R, 0.0)
        return R, -S.sum(1)
    if kind == "coxian":
        return util.coxian_rates(n)
    return util.dense_rates(n, rng, symmetric=(kind == "sym"))


def main():
    po.build()
    assert po.have_ref(), "set PHT_REFERENCE_SRC to an upstream PhaseType source tree to build oracle/_ref"
    cases = [("mhrs_package_y20", "MHRS", "package", 3, 0.0, 2), ("mhrs_dense8_cens", "MHRS", "dense", 8, 0.2, 1),
             ("mhrs_coxian4", "MHRS", "coxian", 4, 0.0, 1), ("dcs_package_y20", "DCS", "package", 3, 0.0, 1),
             ("dcs_sym8", "DCS", "sym", 8, 0.0, 1), ("dcs_coxian4", "DCS", "coxian", 4, 0.0, 1),
             ("ecs_package_y20", "ECS", "package", 3, 0.0, 1), ("ecs_sym8_cens", "ECS", "sym", 8, 0.2, 1),
             ("ecs_coxian4_cens", "ECS", "coxian", 4, 0.3, 1), ("ecs_sym16_cens", "ECS", "sym", 16, 0.2, 1)]
    for name, method, kind, n, fc, mhit in cases:
        rng = np.random.default_rng(abs(hash(name)) % (2 ** 31) if False else sum(map(ord, name)))
        R, s = model(kind, n, rng)
        T, Cm, theta = util.general_model(R, s)
        S, s = util.assemble(T, Cm, theta, n)        # diagonal = sequential row sum, as the reference assembles it
        y = np.array(Y20) if name.endswith("y20") else rng.exponential(1.2, 150) + 0.01
        cens = (rng.uniform(size=y.shape[0]) < fc).astype(np.int32)
        seed, it = 20260000 + n, 3
        out = dict(S=S, s=s, y=y, cens=cens, seed=seed, it=it, mhit=mhit, n=n, method=method)
        if method == "MHRS":
            B, N, z, _ = po.mhrs_paths("ref", seed, it, y, cens, S, s, mhit=mhit)
        else:
            ev, Q, Qi = po.eigen("ref", S, n)
            out.update(evals=ev, Q=Q, Qinv=Qi)
            B, N, z, _ = po.spectral_paths("ref", method, seed, it, y, cens, S, s, spectral=(ev, Q, Qi))
        out.update(B=B, N=N, z=z)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
        print(name, "paths", y.shape[0], "sum N", int(N.sum()), "sum z", float(z.sum()))


if __name__ == "__main__":
    main()
