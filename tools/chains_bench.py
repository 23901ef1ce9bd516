"""Several chains per method-64 engine (pht_engine_set_chains): sweep time of C chains against one, one JSON line per
(shape, C, l).  C3 shape (8 phases, 20 % right-censored) at C in {1, 4, 16, 64, 256} x l in {1e3, 1e4, 1e5, 1e6}, C in
{1, 4} at 1e7, and the C5 shape (32 dense phases) at l = 1e4 for C in {1, 16}.  Per line: ms per sweep (CUDA events
around graph replays of the sweep), chain-sweeps per second (C / ms per sweep), path draws per second (C l per sweep),
and the speed-up over C single-chain engines run one after another (C x the one-chain ms per sweep at the same l, over
this ms per sweep).  The card's name and power limit are printed with every line.
usage: chains_bench.py [OUT.jsonl]   (default: profiles/chains_bench.jsonl; writes there and to stdout)"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import phasetype_b200 as pb
from phasetype_b200 import synth
from phasetype_b200._lib import METHOD_UNIF
from tools.interval_bench import card

WINDOW_MS = 400.0          # timed sweeps are chosen to fill about this much device time


def ms_per_sweep(wl, chains):
    eng = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=METHOD_UNIF, seed=0x5048)
    if chains > 1:
        eng.set_chains(chains)
    eng.set_theta(wl.theta, next_iter=1)
    eng.enqueue(3); eng.sync()                         # warm-up: graph capture, first launches, L2
    total, _ = eng.last_ms()
    steps = int(min(200, max(10, WINDOW_MS / max(total / 3, 1e-3))))
    eng.enqueue(steps); eng.sync()
    total, _ = eng.last_ms()
    eng.close()
    return total / steps, steps


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                               "profiles", "chains_bench.jsonl")
    grid = [("C3", 3, l, (1, 4, 16, 64, 256)) for l in (10 ** 3, 10 ** 4, 10 ** 5, 10 ** 6)]
    grid += [("C3", 3, 10 ** 7, (1, 4)), ("C5 shape, 32 phases", 5, 10 ** 4, (1, 16))]
    name = card()
    with open(out, "w") as f:
        for shape, cfg, l, cs in grid:
            wl = synth.config(cfg, "MHRS", l=l)
            one = None
            for c in cs:
                ms, steps = ms_per_sweep(wl, c)
                if c == 1:
                    one = ms
                rec = {"card": name, "method": 64, "shape": shape, "phases": wl.n, "l": l, "chains": c, "steps": steps,
                       "ms_per_sweep": round(ms, 4), "chain_sweeps_per_s": float("%.4g" % (c / (ms * 1e-3))),
                       "path_draws_per_s": float("%.4g" % (c * l / (ms * 1e-3))),
                       "speedup_vs_separate_engines": round(c * one / ms, 2)}
                line = json.dumps(rec)
                print(line, flush=True)
                f.write(line + "\n")


if __name__ == "__main__":
    main()
