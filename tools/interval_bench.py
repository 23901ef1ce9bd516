"""MHRS sweep time with interval-censored observations: the C3 shape (8 phases, 1e7 observations), with its 20 % of
censored observations inspected on a grid of spacing w (the true absorption time T of each is known to lie in
(floor(T / w) w, floor(T / w) w + w]) instead of right-censored at U T, next to the plain C3 run.  Per run: ms per sweep
(CUDA events around `steps` sweeps replayed from the CUDA graph), path draws per second, rejection attempts run per path,
and, for the interval runs, the attempts the sequential sampler needs per interval observation on average
(1 / P(y <= T <= u) from scipy's expm at the generating rates, where the chain starts).  The card's name and power limit are printed with them.
usage: interval_bench.py [L] [STEPS] [WIDTHS...]     (one JSON line per run)"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import scipy.linalg as sl

import phasetype_b200 as pb
from phasetype_b200 import synth


def c3_with_truth(l):
    """synth.config(3, l=l) together with the absorption times it censored (the same generator draws, in order)."""
    rng = np.random.default_rng(synth.SEED0 + 3)
    R = rng.uniform(0.2, 1.2, (8, 8)); np.fill_diagonal(R, 0.0)
    s = rng.uniform(0.2, 1.2, 8)
    t = synth.simulate_pht(R, s, l, rng)
    flag = rng.random(l) < 0.2
    wl = synth.config(3, "MHRS", l=l)
    assert np.array_equal(wl.censored, flag.astype(np.int32))
    return wl, t, R, s


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return out


def run(wl, u, steps, warmup):
    bounded = u is not None
    sy = float(np.where(np.isfinite(u), u, wl.y).sum()) if bounded else float(wl.y.sum())
    eng = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=1, mhit=1, seed=0x5048, sum_y_global=sy)
    if bounded:
        eng.set_upper(u)
    eng.set_theta(wl.theta, next_iter=1)
    eng.enqueue(warmup); eng.sync()
    c0 = eng.counters()
    eng.enqueue(steps); eng.sync()
    c1 = eng.counters()
    total_ms, _ = eng.last_ms()
    eng.close()
    ms = total_ms / steps
    return {"ms_per_sweep": round(ms, 3), "path_draws_per_s": float("%.4g" % (wl.l / (ms * 1e-3))),
            "attempts_per_path": round((c1["attempts"] - c0["attempts"]) / (steps * wl.l), 3),
            "tail_rounds_per_sweep": round((c1["tail_rounds"] - c0["tail_rounds"]) / steps, 2)}


def expected_attempts(R, s, y, u):
    """mean over the interval observations of 1 / P(y <= T <= u), start in state 0 (few distinct (y, u) on a grid)."""
    S = R.copy(); np.fill_diagonal(S, -(R.sum(1) + s))
    pairs, counts = np.unique(np.stack([y, u], 1), axis=0, return_counts=True)
    surv = {}

    def sv(x):
        if x not in surv:
            surv[x] = sl.expm(S * x)[0].sum()
        return surv[x]
    inv = np.array([1.0 / (sv(a) - sv(b)) for a, b in pairs])
    return float((inv * counts).sum() / counts.sum())


def main():
    l = int(float(sys.argv[1])) if len(sys.argv) > 1 else 10 ** 7
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
    widths = [float(w) for w in sys.argv[3:]] or [1.0, 0.25, 0.05]
    wl, t, R, s = c3_with_truth(l)
    base = {"card": card(), "l": l, "phases": 8, "steps": steps}
    print(json.dumps(dict(base, run="C3, 20 % right-censored", **run(wl, None, steps, 3))), flush=True)
    flag = wl.censored != 0
    for w in widths:
        lo = np.floor(t / w) * w
        y = wl.y.copy(); u = np.full(l, np.inf)
        y[flag] = np.maximum(lo[flag], 1e-12); u[flag] = lo[flag] + w
        wli = synth.Workload(wl.name, wl.n, wl.T, wl.C, wl.theta, wl.nu, wl.zeta, y, wl.censored, wl.R, wl.s)
        res = run(wli, u, steps, 3)
        res["expected_attempts_per_interval_obs"] = round(expected_attempts(R, s, y[flag], u[flag]), 2)
        print(json.dumps(dict(base, run="C3, 20 %% interval-censored, inspection spacing %g" % w, **res)), flush=True)


if __name__ == "__main__":
    main()
