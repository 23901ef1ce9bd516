"""Method 64 with stage visits (Engine.set_stage_visits) on the C3 shape (8 phases, 20 % right-censored): ms per sweep (CUDA
events around `steps` graph replays of the whole sweep) at 1e6 and 1e7 observations, for every observation with y > 0
carrying k in {2, 8, 32} visits at the evenly spaced times j y / (k + 1), read as stage j mod 4 of the 2-phase stages
{2i, 2i+1}.  Three arms per k: the stage masks through set_visits (the panel kernel), the 0/1 indicator E through
set_stage_visits (the emission kernel, E fixed), and a misclassifying E (10 % into each adjacent stage) with a Dirichlet
prior (the emission kernel and the E update).  The card's name and power limit are on every line; lines go to stdout and
to profiles/misclass_bench.jsonl (or the file named by --out).
usage: misclass_bench.py [--sizes 1e6,1e7] [--ks 2,8,32] [--steps S] [--warmup W] [--out FILE]"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import phasetype_b200 as pb
from phasetype_b200 import synth
from phasetype_b200._lib import METHOD_UNIF
from panel_bench import card, visits

STAGE = np.arange(8) // 2
INDICATOR = np.eye(4)[STAGE]
MISREAD = np.array([[0.9, 0.1, 0.0, 0.0], [0.1, 0.8, 0.1, 0.0], [0.0, 0.1, 0.8, 0.1], [0.0, 0.0, 0.1, 0.9]])[STAGE]


def timed(wl, steps, warmup, arm, vis):
    eng = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=METHOD_UNIF, seed=7)
    off, t, stage = vis
    if arm == "masks":
        eng.set_visits(off, t, synth.stage_masks(STAGE)[stage])
    elif arm == "indicator":
        eng.set_stage_visits(INDICATOR, off, t, stage)
    else:
        eng.set_stage_visits(MISREAD, off, t, stage, alpha=np.where(MISREAD > 0, 1.0, 0.0))
    eng.set_theta(wl.theta, next_iter=1)
    eng.run(warmup)
    eng.enqueue(steps)
    eng.sync()
    total, _ = eng.last_ms()
    eng.close()
    return total / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1e6,1e7")
    ap.add_argument("--ks", default="2,8,32")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "misclass_bench.jsonl"))
    a = ap.parse_args()
    gpu = card()
    with open(a.out, "a") as f:
        for size in (int(float(v)) for v in a.sizes.split(",")):
            wl = synth.config(3, "MHRS", l=size)
            for k in (int(v) for v in a.ks.split(",")):
                vis = visits(wl.y, k, lambda j: j % 4)
                for arm in ("masks", "indicator", "misread_prior"):
                    line = json.dumps({"bench": "misclass", "shape": "C3", "l": size, "visits": k, "arm": arm, "steps": a.steps,
                                       "graph": True, "gpu": gpu, "ms_per_sweep": timed(wl, a.steps, a.warmup, arm, vis)})
                    print(line, flush=True)
                    f.write(line + "\n")


if __name__ == "__main__":
    main()
