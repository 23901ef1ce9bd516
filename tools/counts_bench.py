"""Method 64 with counts (Engine.set_counts) against the engine on the expanded data, on the C3 shape (8 phases, 1e7 units).
Per run: ms per sweep (CUDA events around `steps` graph replays of the whole sweep), units per second, and whether the two
engines' theta rows of a few sweeps from the same start are bit-identical.  Workloads:
  (a) fully inspected data (every unit interval- or right-censored on a grid of inspections up to time 8) at spacings 1,
      0.25 and 0.05, tabulated; and the DESIGN mix: 20 % of the units on the 0.25 grid, 80 % exact continuous times;
  (b) exact times rounded to 0.01 with administrative censoring at time 5;
  (c) the plain C3 data (continuous, 20 % right-censored), all counts 1, against the engine without counts;
  (d) a life table of 1e9 units (intervals of 0.1 up to time 8, the rest right-censored there), counts only;
  sweep: the count threshold and the chunk size (PHT_B200_COUNTS_THRESHOLD / _CHUNK) on (b) and on exact times rounded
      to 1e-4 (many records of a few units each).
The card's name and power limit are printed on every line; lines go to stdout and to profiles/counts_bench.jsonl (or the
file named by --out).
usage: counts_bench.py [--l L] [--steps S] [--out FILE] [--only a,b,c,d,sweep]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import scipy.linalg as sl

import phasetype_b200 as pb
from phasetype_b200 import synth
from phasetype_b200._lib import METHOD_UNIF

HORIZON = 8.0


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def c3(l):
    """the C3 workload and the absorption times behind it (the same generator draws, in order)"""
    rng = np.random.default_rng(synth.SEED0 + 3)
    R = rng.uniform(0.2, 1.2, (8, 8)); np.fill_diagonal(R, 0.0)
    s = rng.uniform(0.2, 1.2, 8)
    t = synth.simulate_pht(R, s, l, rng)
    wl = synth.config(3, "MHRS", l=l)
    return wl, t, R, s


def inspected(t, w):
    lo = np.floor(t / w) * w
    late = t > HORIZON
    y = np.where(late, HORIZON, lo)
    u = np.where(late, np.inf, lo + w)
    return y, np.ones(t.shape[0], dtype=np.int32), u


def timed(wl, y, cens, u, counts, steps, warmup, sweeps=3):
    """ms per sweep and the theta rows of `sweeps` sweeps from wl.theta"""
    w = np.ones(y.shape[0]) if counts is None else counts.astype(np.float64)
    top = y if u is None else np.where(np.isfinite(u), u, y)
    sy = float((w * top).sum())
    eng = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, y, cens, method=METHOD_UNIF, seed=0x5048, sum_y_global=sy)
    if u is not None:
        eng.set_upper(u)
    if counts is not None:
        eng.set_counts(counts)
    eng.set_theta(wl.theta, next_iter=1)
    eng.enqueue(warmup); eng.sync()
    eng.enqueue(steps); eng.sync()
    ms = eng.last_ms()[0] / steps
    eng.set_theta(wl.theta, next_iter=1)
    rows = eng.run(sweeps)
    eng.close()
    return ms, rows


def pair(name, wl, y, cens, u, steps, warmup, base, out, tabulate=True):
    """the tabulated records with counts against the engine on their expansion np.repeat(records, counts), which numbers
    the units record by record (the order the contract defines; the original order would give other streams)"""
    units = y.shape[0]
    if tabulate:
        ty, tc, tu, w = synth.tabulate(y, cens, u)
    else:
        ty, tc, tu, w = y, cens, u, np.ones(units, dtype=np.uint32)
    rep = lambda a: None if a is None else np.repeat(a, w)
    ms_e, rows_e = timed(wl, rep(ty), rep(tc), rep(tu), None, steps, warmup)
    ms_c, rows_c = timed(wl, ty, tc, tu, w, steps, warmup)
    line = dict(base, run=name, units=units, records=int(ty.shape[0]), ms_per_sweep_expanded=round(ms_e, 3),
                ms_per_sweep_counts=round(ms_c, 3), units_per_s_expanded=float("%.4g" % (units / (ms_e * 1e-3))),
                units_per_s_counts=float("%.4g" % (units / (ms_c * 1e-3))), speedup=round(ms_e / ms_c, 3),
                bit_identical=bool(np.array_equal(rows_e, rows_c)))
    emit(line, out)


def emit(line, out):
    print(json.dumps(line), flush=True)
    with open(out, "a") as f:
        f.write(json.dumps(line) + "\n")


def life_table(R, s, total, width):
    """expected-count multinomial of `total` units over the intervals (k width, (k+1) width] up to HORIZON, the rest
    right-censored there (start in state 0)"""
    S = R.copy(); np.fill_diagonal(S, -(R.sum(1) + s))
    edges = np.arange(0.0, HORIZON + width / 2, width)
    surv = np.array([sl.expm(S * x)[0].sum() for x in edges])
    p = np.r_[surv[:-1] - surv[1:], surv[-1]]
    w = np.random.default_rng(9).multinomial(total, p / p.sum()).astype(np.uint32)
    y = np.r_[edges[:-1], HORIZON]
    u = np.r_[edges[1:], np.inf]
    return y, np.ones(y.shape[0], dtype=np.int32), u, w


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--l", type=float, default=1e7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "counts_bench.jsonl"))
    ap.add_argument("--only", default="a,b,c,d,sweep")
    a = ap.parse_args()
    only = set(a.only.split(","))
    l = int(a.l)
    wl, t, R, s = c3(l)
    base = {"card": card(), "phases": 8, "steps": a.steps}
    rng = np.random.default_rng(17)
    if "a" in only:
        for w in (1.0, 0.25, 0.05):
            y, c, u = inspected(t, w)
            pair("(a) fully inspected, spacing %g up to %g" % (w, HORIZON), wl, y, c, u, a.steps, a.warmup, base, a.out)
        y, c, u = inspected(t, 0.25)
        grid = rng.random(l) < 0.2
        y = np.where(grid, y, t); c = np.where(grid, 1, 0).astype(np.int32); u = np.where(grid, u, np.inf)
        pair("(a) DESIGN mix: 20 % on the 0.25 grid, 80 % exact continuous", wl, y, c, u, a.steps, a.warmup, base, a.out)
    if "b" in only:
        cens = (t > 5.0).astype(np.int32)
        y = np.where(cens == 1, 5.0, np.maximum(np.round(t, 2), 0.01))
        pair("(b) exact times rounded to 0.01, administrative censoring at 5", wl, y, cens, None, a.steps, a.warmup, base, a.out)
    if "c" in only:
        pair("(c) continuous C3 data, all counts 1", wl, wl.y, wl.censored.astype(np.int32), None, a.steps, a.warmup, base, a.out,
             tabulate=False)
    if "d" in only:
        y, c, u, w = life_table(R, s, 10 ** 9, 0.1)
        ms, rows = timed(wl, y, c, u, w, a.steps, a.warmup)
        emit(dict(base, run="(d) life table of 1e9 units, intervals of 0.1 up to %g, counts only" % HORIZON, units=int(w.astype(np.int64).sum()),
                  records=int(y.shape[0]), ms_per_sweep_counts=round(ms, 3), units_per_s_counts=float("%.4g" % (w.astype(np.int64).sum() / (ms * 1e-3))),
                  finite=bool(np.isfinite(rows).all())), a.out)
    if "sweep" in only:
        cens = (t > 5.0).astype(np.int32)
        for digits in (2, 4):
            y = np.where(cens == 1, 5.0, np.maximum(np.round(t, digits), 10.0 ** -digits))
            ty, tc, tu, w = synth.tabulate(y, cens)
            sy = float((w * ty).sum())
            eng = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, ty, tc, method=METHOD_UNIF, seed=0x5048, sum_y_global=sy)
            ref = None
            for thr in (16, 64, 256, 1024):
                for ch in (32, 64, 128, 256, 1024):
                    os.environ["PHT_B200_COUNTS_THRESHOLD"] = str(thr); os.environ["PHT_B200_COUNTS_CHUNK"] = str(ch)
                    eng.set_counts(w)
                    eng.set_theta(wl.theta, next_iter=1)
                    eng.enqueue(a.warmup); eng.sync()
                    eng.enqueue(a.steps); eng.sync()
                    ms = eng.last_ms()[0] / a.steps
                    eng.set_theta(wl.theta, next_iter=1)
                    rows = eng.run(2)
                    ref = rows if ref is None else ref
                    emit(dict(base, run="sweep: exact times rounded to 1e-%d, administrative censoring at 5" % digits, units=l,
                              records=int(ty.shape[0]), records_at_or_above=int((w >= thr).sum()), threshold=thr, chunk=ch,
                              ms_per_sweep_counts=round(ms, 3), same_as_first=bool(np.array_equal(rows, ref))), a.out)
            eng.close()
            os.environ.pop("PHT_B200_COUNTS_THRESHOLD"); os.environ.pop("PHT_B200_COUNTS_CHUNK")


if __name__ == "__main__":
    main()
