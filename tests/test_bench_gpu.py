"""bench.py --dump-outputs: what it saves is what the last timed sweep computed -- the parameter draw is the last row of
the chain that the warm-up and the `--steps` timed sweeps produce (so `--steps` is the number of sweeps timed), and the
sweep totals and sampled per-observation paths are those of that sweep's iteration, checked against the CPU oracle."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import pyoracle as po

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_is_the_last_timed_sweep(tmp_path):
    import bench
    import phasetype_b200 as pb
    from phasetype_b200 import synth
    cid, method, mhit, l, warmup, steps = 3, "MHRS", 1, 20000, 3, 4
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", str(cid), "--method", method, "--mhit", str(mhit),
                        "--obs", str(l), "--steps", str(steps), "--warmup", str(warmup), "--no-others", "--no-cpu", "--no-e2e",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    d = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert all(a.dtype == np.float64 for a in d.values())
    assert sum(a.nbytes for a in d.values()) <= 64 << 20

    wl = synth.config(cid, method, l=l)
    code = bench.METHOD_CODE[method]
    eng = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=code, mhit=mhit, seed=bench.SEED)
    eng.set_theta(wl.theta, next_iter=1)
    it = warmup + steps                     # the last timed sweep, run from the parameters of the row before it
    prev = eng.run(it - 1)[-1]
    eng.sweep_stats()                       # assembles the generator of that sweep, which model() then reads
    mdl = eng.model()
    last = eng.run(1)[0]
    eng.close()
    assert np.array_equal(d["theta"], last)

    zbits = po.choose_zbits(wl.y.sum())
    N, B, zfix, _ = po.sweep_stats(bench.SEED, it, False, mhit, code, wl.n, wl.T, wl.C, prev, wl.y, wl.censored, zbits=zbits)
    assert np.array_equal(d["sweep_N"], N) and np.array_equal(d["sweep_B"], B)
    assert np.array_equal(d["sweep_z"], zfix * 2.0 ** -zbits)
    W = bench.DUMP_WINDOW
    obs = d["paths_obs"].astype(np.int64)
    assert obs.size > 0 and obs.size % W == 0 and np.unique(obs).size == obs.size
    for k, a in enumerate(obs[::W]):        # windows of W consecutive observations
        assert np.array_equal(obs[k * W:(k + 1) * W], np.arange(a, a + W))
        Bo, No, zo, _ = po.mhrs_paths("oracle", bench.SEED, it, wl.y[a:a + W], wl.censored[a:a + W], mdl["S"], mdl["s"], mhit=mhit,
                                      obs0=int(a))
        rows_w = slice(k * W, (k + 1) * W)
        assert np.array_equal(d["paths_B"][rows_w], Bo) and np.array_equal(d["paths_N"][rows_w], No)
        assert np.array_equal(d["paths_z"][rows_w], zo)
