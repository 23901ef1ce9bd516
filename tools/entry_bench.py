"""Sweep time of the uniformisation sampler (method 64) with delayed entry, one JSON line per run: the C3 shape (8 dense
phases, L observations, 20 % right-censored) where half of the observations carry an entry age a = U min(y, 2) (U uniform
on (0, 1)): about 0.28 units lost before entry per observation at the true parameters.  (Uncapped ages a = U y put some
units at ages where the model leaves almost no survival, which error bit 1024 refuses.)  Reports:
  - ms per sweep with the entry ages, and on the same data with them cleared (CUDA events around `steps` sweeps replayed
    from the CUDA graph, after `warmup` sweeps);
  - ghosts per sweep (the ghost counts of one sweep at the chain's current parameters, at the end of the timed run);
  - the mean durations in microseconds of the entry-table, count and ghost kernels (torch.profiler over a few sweeps
    launched one kernel at a time, in a run of its own).
The card's name and power limit are printed with them.
usage: entry_bench.py [L] [STEPS] [WARMUP]"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import phasetype_b200 as pb
from phasetype_b200._lib import METHOD_UNIF
from tools.interval_bench import c3_with_truth, card

KERNELS = ("k_unif_entry_table", "k_unif_entry_count", "k_unif_ghosts", "k_unif_paths", "k_unif_table")


def _engine(wl, a, sy, use_graph=True):
    eng = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=METHOD_UNIF, seed=0x5048, sum_y_global=sy,
                    use_graph=use_graph)
    if a is not None:
        eng.set_entry(a)
    eng.set_theta(wl.theta, next_iter=1)
    return eng


def kernel_us(wl, a, sy, sweeps=6):
    import warnings

    import torch
    from torch.profiler import ProfilerActivity, profile
    warnings.filterwarnings("ignore", module="torch.profiler")
    torch.cuda.init()
    eng = _engine(wl, a, sy, use_graph=False)
    eng.enqueue(1); eng.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.enqueue(sweeps); eng.sync()
    eng.close()
    out = {}
    for e in prof.key_averages():
        for k in KERNELS:
            if k + "(" in e.key or k + "<" in e.key:
                tot = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                out[k] = round(tot / max(e.count, 1), 1)
    return out


def run(wl, a, sy, steps, warmup):
    eng = _engine(wl, a, sy)
    eng.enqueue(warmup); eng.sync()
    eng.enqueue(steps); eng.sync()
    total_ms, _ = eng.last_ms()
    ghosts = int(eng.entry_paths(paths=False).astype(np.int64).sum()) if a is not None else 0
    eng.close()
    return round(total_ms / steps, 3), ghosts


def main():
    l = int(float(sys.argv[1])) if len(sys.argv) > 1 else 10 ** 7
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
    warmup = int(sys.argv[3]) if len(sys.argv) > 3 else 3
    wl, _, _, _ = c3_with_truth(l)
    rng = np.random.default_rng(0xE17)
    a = np.where(rng.random(l) < 0.5, np.minimum(wl.y, 2.0) * rng.random(l), 0.0)
    sy = float((wl.y + a).sum())
    ms_entry, ghosts = run(wl, a, sy, steps, warmup)
    ms_plain, _ = run(wl, None, sy, steps, warmup)
    line = {"card": card(), "method": 64, "run": "C3, 20 % right-censored, half of the observations with entry age U min(y, 2)",
            "l": l, "phases": 8, "steps": steps, "truncated": int((a > 0).sum()), "ms_per_sweep_entry": ms_entry,
            "ms_per_sweep_no_entry": ms_plain, "ghosts_per_sweep": ghosts, "kernel_us": kernel_us(wl, a, sy)}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
