#!/usr/bin/env python
"""bench.py -- Gibbs-sweep throughput of the B200 engine on BASELINE.json's headline workload.

A "step" is one Gibbs sweep (reference src/PHT_MCMC_Aslett.c:268-405) over all observations: one conditioned
latent-path draw per observation + the conjugate parameter update.  Metric: path draws per second
(= observations x sweeps / time); Gibbs iterations/s is reported beside it.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--method MHRS|ECS|DCS] [--config 3] [--obs L] [--dump-outputs DIR]
  python bench.py --impl reference ...      # the reference's own C on the host cores

Headline: BASELINE.json configs[2] = 8-phase general PHT, 10^7 observations, 20 % right-censored, method MHRS (the
one sampler the reference's phtMCMC() uses); ECS and DCS on the same shape are measured in the same run and reported
under "other_methods".  N > 1: one process per GPU (torchrun) and the SAME 10^7 observations sharded over the N ranks
(observation i -> rank i mod N; "scaling": "strong", as BASELINE's config says).  Per sweep the ranks exchange the
statistics block (NCCL all-reduce inside the captured sweep) and search the deepest part of the MHRS rejection tail
together through peer memory.  The run also checks that every rank's chain is identical and equal to the one-GPU chain
of the same data ("chain_parity"), and times the weak-scaling variant (10^7 observations per GPU) under "weak".

The JSON line carries `roofline` (FP64-issue bound kernel: see DESIGN.md section 5), `cpu_baseline`, `e2e`, `clocks`,
`gpu_launches`.  Only the cpu_baseline / --impl reference legs touch oracle/ (the work model's event counts come from
the kernels' own counters).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METHOD_CODE = {"MHRS": 1, "ECS": 2, "DCS": 4}
SEED = 0x5048B200
FLUSH_BYTES = 256 << 20          # > the 126 MB L2


# ----------------------------------------------------------------------------- work model
def work_per_path(method, n, ev):
    """FP64 instruction-equivalents per path, BASELINE.md section 4 (add/mul/fma/compare = 1, div = 8,
    exp = 20, log = 25), from event counts per path measured on the benchmark's own sweeps."""
    if method == "MHRS":
        return ev["jumps"] * (40 + n) + ev["attempts"] * (n + 2)
    if method == "ECS":
        return ev["jumps"] * (2 * n * n + 55 * n + 715) + ev["dens_evals"] * (23 * n + 26) + 550 * ev["env_updates"]
    if method == "DCS":
        return ev["jumps"] * (n * n + 34 * n + 50) + ev["brent_evals"] * (27 * n + 60) + (2 * n * n + 23 * n)
    raise ValueError(method)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device):
        self.device = device; self.proc = None; self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv"); os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            time.sleep(0.3)          # let the sampler take its first readings before the timed region starts
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 8:
                    continue
                try:
                    sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                   "samples": len(sm), "power_w_max": float(max(power)) if power else None}
        return out


# ----------------------------------------------------------------------------- reference / oracle on the CPU
def _cpu_worker(args):
    """One process = one single-threaded copy of the reference (it is not re-entrant: globals in src/utility.c:8-12)."""
    kind, method, seed, it, y, cens, S, s, mhit, obs0 = args
    from oracle import pyoracle as po
    t0 = time.perf_counter()
    if method == "MHRS":
        po.mhrs_paths(kind, seed, it, y, cens, S, s, mhit=mhit, obs0=obs0, want=False)
    else:
        po.spectral_paths(kind, method, seed, it, y, cens, S, s, obs0=obs0, want=False)
    return time.perf_counter() - t0


def cpu_sweeps(wl, method, mhit, sample, cores, steps, warmup, kind):
    """Time `steps` sweeps of the CPU implementation over the first `sample` observations, split over
    `cores` independent processes.  Returns (paths_per_s, ms_per_step)."""
    import multiprocessing as mp
    S, s = model_matrices(wl)
    y = wl.y[:sample]; c = wl.censored[:sample]
    bounds = np.linspace(0, sample, cores + 1).astype(int)
    ctx = mp.get_context("fork")
    times = []
    with ctx.Pool(cores) as pool:
        for k in range(warmup + steps):
            jobs = [(kind, method, SEED, 1 + k, y[a:b], c[a:b], S, s, mhit, int(a)) for a, b in zip(bounds[:-1], bounds[1:]) if b > a]
            t0 = time.perf_counter()
            pool.map(_cpu_worker, jobs)
            dt = time.perf_counter() - t0
            if k >= warmup:
                times.append(dt)
    tot = float(np.sum(times))
    return sample * steps / tot, 1e3 * tot / steps


def model_matrices(wl):
    n = wl.n
    S = wl.R.copy()
    for i in range(n):
        S[i, i] = -(wl.R[i].sum() + wl.s[i])
    return np.asfortranarray(S).ravel(order="F").copy(), wl.s.copy()


def ref_kind():
    from oracle import pyoracle as po
    po.build()
    return "ref" if po.have_ref() else "oracle"


def ncu_capture(method, l_local, general=False):
    """What the committed `ncu --set full` capture of this workload recorded for the path kernel (profiles/traffic.json,
    written by tools/ncu_traffic.py): DRAM bytes and warp instructions per launch; {} when there is no capture.
    ECS / DCS on the general (unsymmetrised) generator were captured at 4 x 10^6 observations: their per-launch figures are
    scaled by the observation count (both kernels stream the observations once and do per-path work) and say so."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if general:
            for k, v in t.items():
                parts = k.split(":")
                if len(parts) == 3 and parts[0] == method and parts[1] == "general":
                    f = l_local / float(parts[2])
                    c = dict(v)
                    c["dram_bytes_per_launch"] = v["dram_bytes_per_launch"] * f
                    c["warp_instructions_per_launch"] = v["warp_instructions_per_launch"] * f
                    c["source"] = "%s (captured at %s observations, scaled x %.2f)" % (v.get("source"), parts[2], f)
                    return c
        return t.get("%s:%d" % (method, l_local)) or {}
    except Exception:
        return {}


def _peak_hbm():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------- --dump-outputs
DUMP_WINDOW = 256                # observations per sampled window of per-observation paths
DUMP_PATH_BYTES = 32 << 20       # cap on the sampled paths' N array (float64, n*n per observation)


def dump_outputs(path, wl, method, mhit, sum_y, sweeps, theta, device):
    """Save what the last of `sweeps` chain sweeps computed, all float64, so that two builds can be compared output for
    output: theta.npy (m, the parameter draw = the last row Engine.run returns), sweep_N/sweep_B/sweep_z.npy (the sweep's
    totals: N column-major n*n, B n, z n in time units) and, for a fixed seeded sample of observation windows,
    paths_obs.npy (observation index) with paths_B/paths_N/paths_z.npy (each observation's path statistics).
    The totals and paths are recomputed by an untimed one-GPU engine on the whole data set that has run sweeps - 1
    sweeps (the chain does not depend on the number of GPUs); its next sweep must reproduce `theta`."""
    import phasetype_b200 as pb
    e = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=METHOD_CODE[method], mhit=mhit, seed=SEED,
                  device=device, sum_y_global=sum_y)
    e.set_theta(wl.theta, next_iter=1)
    e.run(sweeps - 1)
    N, B, zfix = e.sweep_stats()
    w = min(DUMP_WINDOW, wl.l)
    k = max(1, min(64, wl.l // w, DUMP_PATH_BYTES // (8 * wl.n * wl.n * w)))
    starts = np.sort(np.random.default_rng(SEED).choice(wl.l // w, k, replace=False)) * w
    paths = [e.paths(int(a), w) for a in starts]
    last = e.run(1)[0]
    e.close()
    if not np.array_equal(last, theta):
        raise RuntimeError("the recomputed last sweep does not reproduce the timed chain's parameter draw")
    os.makedirs(path, exist_ok=True)
    out = {"theta": theta, "sweep_N": N, "sweep_B": B, "sweep_z": zfix * 2.0 ** -e.zbits,
           "paths_obs": np.concatenate([np.arange(a, a + w) for a in starts]),
           "paths_B": np.concatenate([p[0] for p in paths]), "paths_N": np.concatenate([p[1] for p in paths]),
           "paths_z": np.concatenate([p[2] for p in paths])}
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


# ----------------------------------------------------------------------------- one measured configuration
class Runner:
    def __init__(self, args, rank, world, local_rank):
        self.a = args; self.rank = rank; self.world = world; self.local_rank = local_rank
        self.torch = None; self.dist = None
        if world > 1:
            import torch
            import torch.distributed as dist
            torch.cuda.set_device(local_rank)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            self.torch = torch; self.dist = dist
            # host-side waits that must not occupy the GPUs (rank 0 drives all devices in the end-to-end leg)
            self.cpu_group = dist.new_group(backend="gloo")

    def barrier(self):
        if self.world > 1:
            self.torch.cuda.synchronize(); self.dist.barrier(); self.torch.cuda.synchronize()

    def host_barrier(self):
        if self.world > 1:
            self.dist.barrier(group=self.cpu_group)

    def chain_parity(self, wl, method, y_loc, c_loc, sum_y, sweeps=3):
        """Every rank's chain must be the same numbers, and the same as the chain ONE GPU draws from the whole data set
        (integer statistics, keyed Philox streams: the number of GPUs must not show in the results)."""
        torch, dist = self.torch, self.dist
        e = self.make_engine(wl, method, y_loc, c_loc, sum_y, True, False)
        rows = e.run(sweeps); e.close()
        mine = torch.from_numpy(rows.copy()).cuda()
        allr = [torch.zeros_like(mine) for _ in range(self.world)]
        dist.all_gather(allr, mine); torch.cuda.synchronize()
        same = all(bool(torch.equal(a, allr[0])) for a in allr)
        ok = torch.zeros(1, dtype=torch.int32, device="cuda")
        if self.rank == 0:
            import phasetype_b200 as pb
            one = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, wl.y, wl.censored, method=METHOD_CODE[method], mhit=self.a.mhit, seed=SEED,
                            device=self.local_rank, rank=0, world=1, use_graph=True, sum_y_global=sum_y)
            one.set_theta(wl.theta, next_iter=1)
            ref = one.run(sweeps); one.close()
            ok[0] = 1 if (same and np.array_equal(ref, rows)) else 0
        dist.broadcast(ok, 0)
        return bool(ok.item())

    def reduce(self, x, op="max"):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return float(t.item())

    def make_engine(self, wl, method, y_loc, c_loc, sum_y, graph, flush):
        import phasetype_b200 as pb
        t0 = time.perf_counter()
        e = pb.Engine(wl.n, wl.T, wl.C, wl.nu, wl.zeta, y_loc, c_loc, method=METHOD_CODE[method], mhit=self.a.mhit, seed=SEED,
                      device=self.local_rank, rank=self.rank, world=self.world, use_graph=graph, sum_y_global=sum_y)
        self.last_create_s = time.perf_counter() - t0          # engine creation = upload of the shard (no communicator yet)
        if self.world > 1:
            torch, dist = self.torch, self.dist
            use_nccl = os.environ.get("PHT_B200_NCCL", "0") not in ("", "0") or bool(os.environ.get("PHT_BENCH_NO_PEERS"))
            if use_nccl:
                # the statistics all-reduce as an ncclAllReduce inside the captured sweep (comparison arm)
                buf = torch.zeros(128, dtype=torch.uint8, device="cuda")
                if self.rank == 0:
                    import ctypes as C
                    raw = (C.c_char * 128)()
                    if pb.lib().pht_comm_unique_id(raw) != 0:
                        raise RuntimeError(pb.lib().pht_last_error().decode())
                    buf.copy_(torch.frombuffer(bytearray(raw.raw), dtype=torch.uint8))
                dist.broadcast(buf, 0)
                e.comm_init(bytes(buf.cpu().numpy().tobytes()))
            if not os.environ.get("PHT_BENCH_NO_PEERS"):
                # the engines' exchange windows (statistics all-reduce + global MHRS tail, both inside the sweep's own
                # kernels): every rank opens every other rank's through CUDA IPC
                from phasetype_b200._lib import PEER_HANDLE_BYTES
                mine = torch.frombuffer(bytearray(e.peer_handle()), dtype=torch.uint8).cuda()
                allh = [torch.zeros(PEER_HANDLE_BYTES, dtype=torch.uint8, device="cuda") for _ in range(self.world)]
                dist.all_gather(allh, mine); torch.cuda.synchronize()
                e.peer_attach(b"".join(bytes(h.cpu().numpy().tobytes()) for h in allh))
        if flush:
            e.set_l2_flush(FLUSH_BYTES)
        e.set_theta(wl.theta, next_iter=1)
        return e

    def timed(self, wl, method, y_loc, c_loc, sum_y, steps, warmup, clocks=False, keep_theta=False):
        """W warm-up sweeps, then exactly `steps` sweeps between barriers; device time from CUDA events on the sweep
        stream, max over ranks.  keep_theta: also return the parameter draw of the last timed sweep.  Returns a dict."""
        eng = self.make_engine(wl, method, y_loc, c_loc, sum_y, True, True)
        eng.run(warmup)
        c0 = eng.counters()
        sampler = ClockSampler(self.local_rank) if (clocks and self.rank == 0) else None
        if sampler:
            sampler.start()
        self.barrier()
        t0 = time.perf_counter()
        eng.enqueue(steps); eng.sync()
        wall = time.perf_counter() - t0
        self.barrier()
        clk = sampler.stop() if sampler else None
        total_ms, _ = eng.last_ms()
        total_ms = self.reduce(total_ms)
        c1 = eng.counters()
        theta = eng.get_theta() if keep_theta else None
        eng.close()
        # instrumented pass: duration of the path kernel alone (CUDA events around each launch, no graph)
        eng2 = self.make_engine(wl, method, y_loc, c_loc, sum_y, False, True)
        eng2.run(warmup)
        self.barrier()
        k = min(steps, 32)
        eng2.enqueue(k); eng2.sync()
        tot2, kern_ms = eng2.last_ms()
        if os.environ.get("PHT_BENCH_VERBOSE"):
            cc = eng2.counters()
            sys.stderr.write("rank %d: path kernels %.3f ms/sweep (lanes %.2f, local tail %.2f, global tail %.2f, replay kernel %.2f ms), %d observations handed to the tail, %.1f tail rounds per sweep\n"
                             % (self.rank, kern_ms, cc["ns_lane"] * 1e-6 / (warmup + k), cc["ns_tail"] * 1e-6 / (warmup + k), cc["ns_global"] * 1e-6 / (warmup + k),
                                cc["ns_replay"] * 1e-6 / (warmup + k), cc["deferred"] // (warmup + k), cc["tail_rounds"] / float(warmup + k)))
        kern_ms = self.reduce(kern_ms)
        eng2.close()
        nloc = max(1, y_loc.shape[0])
        return {"total_ms": total_ms, "wall": wall, "clocks": clk, "launches": int(c1["launches"] - c0["launches"]), "theta": theta,
                "kern_ms": kern_ms, "share": kern_ms * k / max(tot2, 1e-9),
                "events": {q: (c1[q] - c0[q]) / float(steps * nloc) for q in ("attempts", "jumps", "deferred", "dens_evals", "env_updates", "brent_evals")},
                "tail_rounds": (c1["tail_rounds"] - c0["tail_rounds"]) / float(steps)}

    def roofline(self, wl, method, res, l_local, fma_rate):
        # events per path counted by the kernels themselves over the timed sweeps (every attempt and jump-step the GPU
        # ran, including the replay of accepted attempts): the work model needs nothing from the CPU checker
        ev = res["events"]
        W = work_per_path(method, wl.n, ev)
        achieved = W * l_local / (res["kern_ms"] * 1e-3)
        hbm_peak, hbm_src = _peak_hbm()
        kernel = {"MHRS": "k_mhrs_lanes + k_mhrs_tail + k_mhrs_replay", "DCS": "k_dcs_sweep", "ECS": "k_ecs_exact + k_ecs_gt"}[method]
        cap = ncu_capture(method, l_local, general=(method != "MHRS" and "symmetric" not in wl.name and wl.name.startswith("C3")))
        issue = None
        mhz = (res.get("clocks") or {}).get("sm_mhz") or getattr(self, "sm_mhz", None)
        if cap.get("warp_instructions_per_launch") and mhz:
            # second view of the same kernel: share of the SMs' warp-instruction issue slots it fills (148 SMs x 4 schedulers
            # x clock); instruction count from the committed capture, time and clock from this run
            slots = res["kern_ms"] * 1e-3 * 148 * 4 * mhz * 1e6
            issue = {"warp_instructions_per_launch": cap["warp_instructions_per_launch"], "issue_slot_utilisation": cap["warp_instructions_per_launch"] / slots,
                     "active_lanes_per_instruction": cap.get("active_lanes_per_instruction"), "source": cap.get("source")}
        return {"bound": "fp64_issue", "achieved": achieved / 1e9, "peak": fma_rate / 1e9, "unit": "G FP64-instr-equiv/s",
                "frac": achieved / fma_rate, "traffic": cap.get("dram_bytes_per_launch"), "issue": issue,
                "traffic_and_issue": "from_capture: read from the committed ncu capture %s, not measured in this run" % cap.get("source") if cap else None,
                "peak_source": "measured in this run: dependent FP64 FMA chains on all SMs (pht_fp64_fma_rate); burst figure",
                "kernel": kernel, "kernel_ms": res["kern_ms"], "kernel_share_of_step": res["share"],
                "work_per_path": W, "events_per_path": ev,
                "hbm": {"algorithmic_bytes_per_launch": 9 * l_local, "achieved_GBs": 9e-9 * l_local / (res["kern_ms"] * 1e-3),
                        "peak_GBs": hbm_peak, "peak_source": hbm_src,
                        # MHRS streams more than the 9 B per path of the observation itself BY DESIGN: the search kernels read y, flag and
                        # the sort permutation (13 B) and write a 16-byte record, which the replay kernel reads back with y, flag and
                        # permutation (29 B): 58 B per path, ~0.05 ms of HBM time in a sweep of > 10 ms (DESIGN.md section 3)
                        "streamed_by_design_bytes_per_launch": (58 if method == "MHRS" else 9) * l_local}}


# ----------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--method", default="MHRS", choices=["MHRS", "ECS", "DCS"])
    ap.add_argument("--config", type=int, default=3)
    ap.add_argument("--obs", dest="l", type=int, default=None, help="observations per GPU (default: the config's own count)")
    ap.add_argument("--mhit", type=int, default=1)
    ap.add_argument("--cpu-sample", type=int, default=None)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="skip the ECS / DCS side measurements at N = 1")
    ap.add_argument("--no-weak", action="store_true", help="skip the weak-scaling side measurement at N > 1")
    ap.add_argument("--no-parity", action="store_true", help="skip the chain-parity check at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="save what the last timed sweep computed as DIR/<name>.npy (parameter draw, sweep totals, a fixed "
                         "sample of per-observation paths) so that two builds can be compared on the same seeded inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 arm (the reference arm keeps no outputs)")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    from phasetype_b200 import synth
    full_l = args.l or {1: 100, 2: 10 ** 6, 3: 10 ** 7, 4: 10 ** 7, 5: 10 ** 8}[args.config]

    if args.impl == "reference":
        if rank != 0:
            return 0
        wl = synth.config(args.config, args.method, l=min(full_l, 2 * 10 ** 6))
        cores = os.cpu_count() or 1
        kind = ref_kind()
        sample = args.cpu_sample or min(wl.l, 20000 * cores)
        pps, ms = cpu_sweeps(wl, args.method, args.mhit, sample, cores, args.steps, args.warmup, kind)
        line = {"impl": "reference", "metric": "path_draws_per_sec", "value": pps, "unit": "paths/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "gibbs_iters_per_sec_extrapolated": pps / full_l,
                "config": {"workload": wl.name, "method": args.method, "mhit": args.mhit, "phases": wl.n,
                           "observations": full_l, "sample_per_step": sample},
                "cpu_baseline": {"value": pps, "unit": "paths/s", "cores": cores,
                                 "kind": "reference" if kind == "ref" else "port",
                                 "sample": "%d observations per step, %d single-threaded processes (the reference is single-threaded and not re-entrant)" % (sample, cores)},
                "e2e": {"value": pps, "unit": "paths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ B200 arm
    import phasetype_b200 as pb
    R = Runner(args, rank, world, local_rank)
    method = args.method
    # the config's own data set, the same on every rank; rank r works on observations r, r + N, ...
    wl = synth.config(args.config, method, l=full_l)
    if world > 1:
        ys, cs = wl.shard(rank, world)
        y_loc = np.ascontiguousarray(ys); c_loc = np.ascontiguousarray(cs)
    else:
        y_loc = np.ascontiguousarray(wl.y); c_loc = np.ascontiguousarray(wl.censored)
    l_local = int(y_loc.shape[0]); l_global = wl.l
    sum_y = float(wl.y.sum())

    res = R.timed(wl, method, y_loc, c_loc, sum_y, args.steps, args.warmup, clocks=True, keep_theta=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, wl, method, args.mhit, sum_y, args.warmup + args.steps, res["theta"], local_rank)
    R.sm_mhz = (res.get("clocks") or {}).get("sm_mhz")
    value = l_global * args.steps / (res["total_ms"] * 1e-3)

    line = None
    if rank == 0:
        fma_rate = pb.fp64_fma_rate(local_rank)
        line = {"metric": "path_draws_per_sec", "value": value, "unit": "paths/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["total_ms"] / args.steps,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "gibbs_iters_per_sec": args.steps / (res["total_ms"] * 1e-3),
                "config": {"workload": wl.name, "method": method, "mhit": args.mhit, "phases": wl.n, "parameters": wl.m,
                           "observations": l_global, "observations_per_gpu": l_local,
                           "sharding": "observation i of the %d -> rank i mod %d; per sweep one all-reduce of n^2+3n+1 int64 (%s) and the global MHRS tail over peer memory" % (l_global, world, "ncclAllReduce" if os.environ.get("PHT_B200_NCCL", "0") not in ("", "0") else "k_allreduce_peer: NVLink peer stores + flag barrier, no library call")
                           if world > 1 else "single GPU",
                           "l2": "flushed: a %d MiB memset on the sweep stream before every sweep, inside the timed region" % (FLUSH_BYTES >> 20)},
                "gpu_launches": res["launches"], "wall_ms_per_step": 1e3 * res["wall"] / args.steps,
                "device_events_per_path": res["events"], "tail_rounds_per_sweep": res["tail_rounds"],
                "clocks": res["clocks"]}
        line["roofline"] = R.roofline(wl, method, res, l_local, fma_rate)

    # ---- N > 1: the chain must not depend on the number of GPUs
    if world > 1 and not args.no_parity:
        ok = R.chain_parity(wl, method, y_loc, c_loc, sum_y)
        if rank == 0:
            line["chain_parity"] = ok
        if not ok:
            sys.stderr.write("rank %d: CHAIN PARITY FAILED: the %d-GPU chain differs between ranks or from the 1-GPU chain\n" % (rank, world))

    # ---- weak scaling beside it (N > 1): every rank its own 10^7 observations of the same model
    if world > 1 and not args.no_weak:
        wlw = synth.config(args.config, method, l=full_l, shard=rank)
        sum_w = R.reduce(float(wlw.y.sum()), "max") * world * 1.0000001
        rw = R.timed(wlw, method, np.ascontiguousarray(wlw.y), np.ascontiguousarray(wlw.censored), sum_w, args.steps, args.warmup)
        if rank == 0:
            line["weak"] = {"observations": full_l * world, "value": full_l * world * args.steps / (rw["total_ms"] * 1e-3), "unit": "paths/s",
                            "ms_per_step": rw["total_ms"] / args.steps, "kernel_ms": rw["kern_ms"]}
        del wlw

    # ---- the two BASELINE shapes that are 8-GPU jobs as stated (config 4: 10^7 observations, ECS; config 5: 10^8
    # observations, 32 phases): sharded over the ranks like the headline.  Every rank simulates its own shard (an
    # independent stream of the same model); for C5 it simulates 2.5 x 10^6 observations and tiles them to its share --
    # the paths still differ, they are keyed by the global observation index -- because simulating 10^8 32-phase
    # absorption times on the host would take longer than the whole bench.
    if world >= int(os.environ.get("PHT_BENCH_BIGCFG_MIN_WORLD", "8")) and args.config == 3 and not args.no_others:
        oc = {}
        for cid, m2, l2, sim in ((4, "ECS", 10 ** 7, None), (5, "MHRS", 10 ** 8, 2500000)):
            per = l2 // world
            wc = synth.config(cid, m2, l=min(per, sim or per), shard=rank)
            reps = -(-per // wc.l)
            yc = np.ascontiguousarray(np.tile(wc.y, reps)[:per]); cc = np.ascontiguousarray(np.tile(wc.censored, reps)[:per])
            sum_c = R.reduce(float(yc.sum()), "max") * world * 1.0000001
            r2 = R.timed(wc, m2, yc, cc, sum_c, 3, 3)
            if rank == 0:
                rf = R.roofline(wc, m2, r2, per, pb.fp64_fma_rate(local_rank))
                oc["C%d:%s" % (cid, m2)] = {"value": per * world * 3 / (r2["total_ms"] * 1e-3), "unit": "paths/s", "ms_per_step": r2["total_ms"] / 3,
                                            "workload": wc.name, "phases": wc.n, "parameters": wc.m, "observations": per * world,
                                            "observations_per_gpu": per, "simulated_per_gpu": wc.l, "steps": 3, "warmup": 3,
                                            "roofline": {k: rf[k] for k in ("bound", "achieved", "peak", "unit", "frac", "kernel", "kernel_ms", "work_per_path")}}
            del wc, yc, cc
        if rank == 0:
            line["other_configs"] = oc

    # ---- end to end through the drop-in routine with host buffers (upload, communicator set-up, sweeps, download)
    e2e = None
    if not args.no_e2e:
        R.barrier()
        code = METHOD_CODE[method]
        dt = 0.0
        if rank == 0:
            # ONE call of LJMA_Gibbs, as R makes it: the routine itself fans out over the N devices (host threads, NCCL
            # communicator, peer windows); the other ranks of this launch keep their GPUs idle meanwhile
            os.environ["PHT_B200_SEED"] = str(SEED); os.environ["PHT_B200_QUIET"] = "1"
            os.environ["PHT_B200_DEVICE"] = str(local_rank if world == 1 else 0); os.environ["PHT_B200_GPUS"] = str(world)
            dts = []
            # two untimed calls first, like the warm-up sweeps of the device-timed figure: the first call of a process creates
            # the CUDA contexts of the devices it fans out over (seconds) and fills their memory pools; then the median of three
            for rep in range(5):
                t0 = time.perf_counter()
                out = pb.ljma_gibbs(args.steps + 1, args.mhit, code, wl.n, wl.m, wl.nu, wl.zeta, wl.T, wl.C, wl.y,
                                    wl.censored, wl.theta, silent=True)
                if rep >= 2:
                    dts.append(time.perf_counter() - t0)
                assert np.isfinite(out).all() and (out[1:] > 0).all()
            dt = float(np.median(dts))
        R.host_barrier()
        e2e = {"value": l_global * args.steps / dt if dt > 0 else None, "unit": "paths/s", "h2d_bytes_per_step": int(12 * l_global / args.steps),
               "d2h_bytes_per_step": int(8 * wl.m), "seconds": dt, "runs": 3, "warmup_calls": 2,
               "note": "one LJMA_Gibbs(it=%d) call on host vectors driving %d GPU(s): engine creation, upload of y/censored (once per call, amortised over "
                       "the sweeps), %s%d sweeps, download of res" % (args.steps + 1, world, "peer-window set-up (no NCCL in the call), " if world > 1 else "", args.steps)}
    if rank == 0:
        line["e2e"] = e2e
        # ---- the other two samplers on the same shape (N = 1 only; fewer sweeps)
        if world == 1 and not args.no_others:
            # ECS and DCS run on the headline workload itself (general dense S: sweeps whose generator has complex eigenvalue
            # pairs go through the real block form of the spectral formulas -- for DCS the CPLX instance of the same
            # unit-machine kernel); "DCS:symmetric" is DCS on the symmetrised variant of the same shape, where every
            # sweep runs the reference's own arithmetic
            others = {}
            for m2, sym in (("ECS", False), ("DCS", False), ("DCS", True)):
                if m2 == method:
                    continue
                wl_sym = synth.config(args.config, m2 if sym else "MHRS", l=full_l)
                c2 = np.ascontiguousarray(wl_sym.censored if m2 != "DCS" else np.zeros_like(wl_sym.censored))
                r2 = R.timed(wl_sym, m2, np.ascontiguousarray(wl_sym.y), c2, float(wl_sym.y.sum()), 5, 3)
                rf = R.roofline(wl_sym, m2, r2, wl_sym.l, fma_rate)
                others[m2 + (":symmetric" if sym else "")] = {"value": wl_sym.l * 5 / (r2["total_ms"] * 1e-3), "unit": "paths/s", "ms_per_step": r2["total_ms"] / 5,
                              "workload": wl_sym.name, "steps": 5, "warmup": 3, "gpu_launches": r2["launches"],
                              "roofline": {k: rf[k] for k in ("bound", "achieved", "peak", "unit", "frac", "traffic", "issue", "kernel", "kernel_ms", "work_per_path")}}
                del wl_sym
            line["other_methods"] = others
            # ---- the other BASELINE shapes, each at the size BASELINE.json states for one GPU's share (fewer sweeps):
            # C2 = 4-phase Coxian, 10^6 exact observations; C4 = 16-phase tied-rate reliability structure, 10^7
            # observations, ECS (its stated sampler; MHRS cannot sample observations whose survival probability is below
            # 2^-32 and reports that); C5 = 32-phase general PHT: one GPU's share of a 2 x 10^7 slice (the full 10^8 is an
            # 8-GPU job: profiles/r2_configs.md)
            if args.config == 3:
                oc = {}
                # (C5 under ECS / DCS: the general 32-phase generator -- complex spectra, block formulas -- on a 10^5-observation
                # sample: a sweep of the stated 10^8 observations is a minute of one GPU under these samplers)
                for cid, m2, l2 in ((2, "MHRS", 10 ** 6), (2, "ECS", 10 ** 6), (2, "DCS", 10 ** 6), (4, "ECS", 10 ** 7), (5, "MHRS", 2500000),
                                    (5, "ECS", 10 ** 5), (5, "DCS", 10 ** 5)):
                    wc = synth.config(cid, "MHRS" if cid == 5 else m2, l=l2)
                    r2 = R.timed(wc, m2, np.ascontiguousarray(wc.y), np.ascontiguousarray(wc.censored), float(wc.y.sum()), 5, 3)
                    rf = R.roofline(wc, m2, r2, wc.l, fma_rate)
                    oc["C%d:%s" % (cid, m2)] = {"value": wc.l * 5 / (r2["total_ms"] * 1e-3), "unit": "paths/s", "ms_per_step": r2["total_ms"] / 5,
                                                "workload": wc.name, "phases": wc.n, "parameters": wc.m, "observations": wc.l, "steps": 5, "warmup": 3,
                                                "gpu_launches": r2["launches"],
                                                "roofline": {k: rf[k] for k in ("bound", "achieved", "peak", "unit", "frac", "kernel", "kernel_ms", "work_per_path")}}
                    del wc
                line["other_configs"] = oc
        if not args.no_cpu:
            from oracle import pyoracle as po
            po.build()
            kind = "ref" if po.have_ref() else "oracle"
            sample = args.cpu_sample or min(l_local, 100000)
            pps, ms = cpu_sweeps(wl, method, args.mhit, sample, 1, 3, 1, kind)
            line["cpu_baseline"] = {"value": pps, "unit": "paths/s", "cores": 1,
                                    "kind": "reference" if kind == "ref" else "port",
                                    "sample": "first %d observations of the workload, 3 sweeps, 1 process (the reference is single-threaded)" % sample}
        print(json.dumps(line))
    if world > 1:
        R.dist.barrier(); R.dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
