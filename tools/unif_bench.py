"""Sweep time of the uniformisation sampler (method 64) on the shapes it was built for, one JSON line per run:
  - C3 (8 phases, 1e7 observations) with its 20 % censored observations right-censored;
  - C3 with them interval-censored on inspection grids of spacing 1 / 0.25 / 0.05 (as tools/interval_bench.py builds them);
  - C5's shape (32 dense phases) at L5 observations;
  - a tied Coxian (4 phases, forward rate 1.5, exit rate 0.3 from every phase: a Jordan block) at 1e7 exact observations.
Per run: ms per sweep (CUDA events around `steps` sweeps replayed from the CUDA graph), path draws per second, and the
table kernel's mean duration in microseconds (torch.profiler over a few sweeps launched one kernel at a time, in a run
of its own).  The card's name and power limit are printed with them.
usage: unif_bench.py [L] [STEPS] [L5]"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import phasetype_b200 as pb
from phasetype_b200 import synth
from phasetype_b200._lib import METHOD_UNIF
from tools.interval_bench import c3_with_truth, card


def table_us(wl, u, sweeps=6):
    import warnings

    import torch
    from torch.profiler import ProfilerActivity, profile
    warnings.filterwarnings("ignore", module="torch.profiler")        # keep stdout / stderr free of its cycle notice
    torch.cuda.init()
    eng = _engine(wl, u, use_graph=False)
    eng.enqueue(1); eng.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.enqueue(sweeps); eng.sync()
    eng.close()
    ev = [e for e in prof.key_averages() if "k_unif_table" in e.key]
    if not ev:
        return None
    e = ev[0]
    tot = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
    return round(tot / max(e.count, 1), 1)


def _engine(wl, u, use_graph=True):
    sy = float(np.where(np.isfinite(u), u, wl.y).sum()) if u is not None else float(wl.y.sum())
    eng = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=METHOD_UNIF, seed=0x5048, sum_y_global=sy,
                    use_graph=use_graph)
    if u is not None:
        eng.set_upper(u)
    eng.set_theta(wl.theta, next_iter=1)
    return eng


def run(wl, u, steps, warmup=3):
    eng = _engine(wl, u)
    eng.enqueue(warmup); eng.sync()
    eng.enqueue(steps); eng.sync()
    total_ms, _ = eng.last_ms()
    eng.close()
    ms = total_ms / steps
    return {"ms_per_sweep": round(ms, 3), "path_draws_per_s": float("%.4g" % (wl.l / (ms * 1e-3))),
            "table_us": table_us(wl, u)}


def tied_coxian(l):
    n = 4
    R = np.diag(np.full(n - 1, 1.5), 1); s = np.full(n, 0.3)
    Tm = np.zeros((n + 1, n + 1), dtype=np.int32)
    for i in range(n - 1):
        Tm[i, i + 1] = 1
    Tm[:n, n] = 2
    theta = np.array([1.5, 0.3])
    y = synth.simulate_pht(R, s, l, np.random.default_rng(synth.SEED0 + 64))
    return synth.Workload("tied Coxian, 4 phases", n, Tm.ravel(order="F").copy(), np.ones((n + 1) ** 2), theta,
                          np.full(2, 2.0), 2.0 / theta, y, np.zeros(l, dtype=np.int32), R, s)


def main():
    l = int(float(sys.argv[1])) if len(sys.argv) > 1 else 10 ** 7
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
    l5 = int(float(sys.argv[3])) if len(sys.argv) > 3 else 10 ** 7
    base = {"card": card(), "method": 64, "steps": steps}
    wl, t, _, _ = c3_with_truth(l)
    print(json.dumps(dict(base, run="C3, 20 % right-censored", l=l, phases=8, **run(wl, None, steps))), flush=True)
    flag = wl.censored != 0
    for w in (1.0, 0.25, 0.05):
        lo = np.floor(t / w) * w
        y = wl.y.copy(); u = np.full(l, np.inf)
        y[flag] = lo[flag]; u[flag] = lo[flag] + w                  # y = 0 below the first inspection: left-censored
        wli = synth.Workload(wl.name, wl.n, wl.T, wl.C, wl.theta, wl.nu, wl.zeta, y, wl.censored, wl.R, wl.s)
        print(json.dumps(dict(base, run="C3, 20 %% interval-censored, inspection spacing %g" % w, l=l, phases=8,
                              **run(wli, u, steps))), flush=True)
    w5 = synth.config(5, "MHRS", l=l5)
    print(json.dumps(dict(base, run="C5 shape, 32 dense phases", l=l5, phases=32, **run(w5, None, steps))), flush=True)
    wt = tied_coxian(l)
    print(json.dumps(dict(base, run="tied Coxian (F = 1.5, R = 0.3), exact", l=l, phases=4, **run(wt, None, steps))), flush=True)


if __name__ == "__main__":
    main()
