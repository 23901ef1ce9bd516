"""Method 64 with visits (Engine.set_visits) on the C3 shape (8 phases, 20 % right-censored): ms per sweep (CUDA events around
`steps` graph replays of the whole sweep) at 1e6 and 1e7 observations, for every observation with y > 0 carrying k in
{2, 8, 32} visits at the evenly spaced times j y / (k + 1), with singleton masks (the phase j mod 8) or with the 2-phase
stage masks {2i, 2i+1} (stage j mod 4), against the same data without visits.  The card's name and power limit are on
every line; lines go to stdout and to profiles/panel_bench.jsonl (or the file named by --out).
usage: panel_bench.py [--sizes 1e6,1e7] [--ks 2,8,32] [--steps S] [--warmup W] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import phasetype_b200 as pb
from phasetype_b200 import synth
from phasetype_b200._lib import METHOD_UNIF


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def visits(y, k, masks):
    """k evenly spaced visits inside (0, y) for every observation with y > 0; masks(j) gives visit j's mask"""
    has = y > 0
    offsets = np.concatenate([[0], np.cumsum(np.where(has, k, 0))]).astype(np.int64)
    j = np.tile(np.arange(1, k + 1), int(has.sum()))
    t = np.repeat(y[has], k) * j / (k + 1.0)
    return offsets, t, masks(j - 1).astype(np.uint32)


def timed(wl, steps, warmup, vis=None):
    eng = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=METHOD_UNIF, seed=7)
    if vis is not None:
        eng.set_visits(*vis)
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
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "panel_bench.jsonl"))
    a = ap.parse_args()
    gpu = card()
    kinds = {"singleton": lambda j: 1 << (j % 8), "stage2": lambda j: 3 << (2 * (j % 4))}
    with open(a.out, "a") as f:
        for size in (int(float(v)) for v in a.sizes.split(",")):
            wl = synth.config(3, "MHRS", l=size)
            rows = [{"visits": 0, "masks": None, "ms_per_sweep": timed(wl, a.steps, a.warmup)}]
            for k in (int(v) for v in a.ks.split(",")):
                for name, fn in kinds.items():
                    rows.append({"visits": k, "masks": name, "ms_per_sweep": timed(wl, a.steps, a.warmup, visits(wl.y, k, fn))})
            for r in rows:
                line = json.dumps(dict({"bench": "panel", "shape": "C3", "l": size, "steps": a.steps, "graph": True, "gpu": gpu}, **r))
                print(line, flush=True)
                f.write(line + "\n")


if __name__ == "__main__":
    main()
