"""Groups with their own structure per method-64 engine (pht_engine_set_groups): sweep time of a grouped engine against the
ungrouped engine on the same data, one JSON line per case.
  - C3 shape (8 dense phases, 20 % right-censored) at l = 1e7, observation k in group k mod G for G in {1, 2, 8, 32},
    against the ungrouped C3 engine on the same data (G = 0 in the output).  Every group's structure is C3's (its own
    copy of the cells over C3's 64 parameters), so the path work equals C3's by construction and the difference is the
    cost of grouping itself: the grouped layout, G tables, the walking path kernel and the gather over groups.  (Exit
    parameters of each group's own do not fit at G = 32: an engine takes at most n(n+1) = 72 parameters.);
  - the same shape at l = 1e4 with G = 8 and 16 chains, against 16 ungrouped chains and one grouped chain.
Per line: ms per sweep (CUDA events around graph replays), and from a run with direct launches the path kernel's ms per
sweep and the rest (assembly, the G x chains table builds, the update).  The card's name and power limit are printed with
every line.
usage: groups_bench.py [OUT.jsonl]   (default: profiles/groups_bench.jsonl; writes there and to stdout)"""
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


def c3_groups(wl, G):
    """C3's structure once per group: (T, C) of shape (G, (n+1)^2) and theta (C3's)."""
    return np.tile(np.asarray(wl.T, dtype=np.int32), (G, 1)), np.tile(np.asarray(wl.C, dtype=np.float64), (G, 1)), wl.theta


def measure(wl, G, chains):
    """(ms per sweep with graph replays, path-kernel ms per sweep and the rest from direct launches)."""
    out = []
    for graph in (True, False):
        if G:
            T, C, theta = c3_groups(wl, G)
        else:
            T, C, theta = wl.T, wl.C, wl.theta
        m = theta.shape[0]
        eng = pb.Engine(wl.n, T[0] if G else T, C[0] if G else C, np.full(m, 2.0), 2.0 / theta, wl.y, wl.censored,
                        method=METHOD_UNIF, seed=0x5048, use_graph=graph)
        if chains > 1:
            eng.set_chains(chains)
        if G:
            eng.set_groups(T, C, (np.arange(wl.l) % G).astype(np.int32))
        eng.set_theta(theta, next_iter=1)
        eng.enqueue(3); eng.sync()                     # warm-up: graph capture, first launches, L2
        total, _ = eng.last_ms()
        steps = int(min(200, max(10, WINDOW_MS / max(total / 3, 1e-3))))
        eng.enqueue(steps); eng.sync()
        total, path = eng.last_ms()
        eng.close()
        out.append((total / steps, path, steps))
    return out[0][0], out[1][1], out[1][0] - out[1][1], out[0][2]


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                               "profiles", "groups_bench.jsonl")
    name = card()
    cases = [(10 ** 7, G, 1) for G in (0, 1, 2, 8, 32)] + [(10 ** 4, G, c) for G, c in ((0, 16), (8, 1), (8, 16))]
    wls = {}
    with open(out, "w") as f:
        seen = {}
        for l, G, chains in cases:
            if l not in wls:
                wls[l] = synth.config(3, "MHRS", l=l)
            ms, path_ms, rest_ms, steps = measure(wls[l], G, chains)
            seen[(l, G, chains)] = ms
            ungrouped, one = seen.get((l, 0, chains)), seen.get((l, G, 1))
            rec = {"card": name, "method": 64, "shape": "C3", "phases": 8, "l": l, "groups": G, "chains": chains, "steps": steps,
                   "ms_per_sweep": round(ms, 4), "direct_path_kernel_ms": round(path_ms, 4), "direct_rest_ms": round(rest_ms, 4),
                   "vs_ungrouped_same_chains": round(ms / ungrouped, 4) if G and ungrouped else None,
                   "vs_one_chain": round(ms / one, 4) if chains > 1 and one else None}
            line = json.dumps(rec)
            print(line, flush=True)
            f.write(line + "\n")


if __name__ == "__main__":
    main()
