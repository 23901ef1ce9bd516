/*
 * k_mhrs.cu -- Bladt MHRS path sampler for sm_100a (method bit 1).
 *
 * What it computes (reference: per-observation independence Metropolis-Hastings over
 * rejection-sampled paths, src/Simulate_AbsCTMC_eq_Bladt_MHRS.c:63-110 calling
 * src/Simulate_AbsCTMC_gt_Bladt_MHRS.c:34-160): for every observation y, forward-simulate
 * the unconditioned chain until an attempt survives past y, optionally MH-swap against
 * `mhit` further draws, and add the accepted path's (B, N, z) to the sweep statistics.
 *
 * How it is organised on the GPU (nothing like the reference's loop nest):
 *   - Every rejection attempt is its own Philox sub-stream (pht_philox.h), so attempts are
 *     independent work items and "the first attempt that survives" is well defined whatever
 *     order, lane or GPU they run on.
 *   - SEARCH / REPLAY split.  ~21 of 22 attempts fail, and a failed attempt contributes
 *     nothing but the fact that it failed.  The search therefore runs a FILTER walk: the state
 *     sequence is exact (the scan `while (sofar < target) sofar += p[k++]` is answered by
 *     integer thresholds on the 52 random bits -- same decisions as the FP64 comparison), but
 *     the clock is kept in FP32 with the exponential taken from MUFU.LG2, together with a
 *     rigorous bound of its error.  "Attempt alive at y?" is decided by the filter when the
 *     clock is further from y than the bound; the rare attempt that ends inside the band
 *     (~1e-4 of them) is re-run by the exact FP64 walker.  The decision is therefore always
 *     the exact one, at a third of the instructions.  The accepted attempt is replayed once
 *     by the exact walker with recording on: every N, B and z bit comes from FP64 arithmetic
 *     in the reference's order.
 *   - One jump-step is one Philox block: {state uniform of this jump, exponential uniform of
 *     the next sojourn}.  A failed attempt restarts the lane on the next sub-stream with a
 *     handful of selects, so fresh, running and failing lanes execute one instruction stream.
 *   - Lane phase: persistent warps, one observation per lane.  Observations are laid out by
 *     decreasing y (the attempt count is Geometric(survival(y))), so the stream ends with the
 *     cheapest observations and the drain is short.  Every lane holds one prefetched
 *     observation; empty slots are refilled eight or more at a time from a global counter.
 *     A finished observation leaves a 16-byte RECORD (its one or two surviving attempts and the
 *     end states the accept test needs) in a list indexed by its position; the replay is the
 *     third kernel's business.
 *   - A lane gives up after `cap` attempts (attempt counts have a heavy tail, SURVEY.md H2) and
 *     appends the observation to the tail list.
 *   - Tail phase (same cooperative launch, grid barriers between rounds): the attempts of every
 *     pending observation are searched by all warps of the GPU.  A warp takes a pool of
 *     consecutive attempts of ONE observation from a global counter, its lanes draw attempt
 *     indices from the pool with a ballot, the lowest surviving attempt wins through atomicMin;
 *     one thread per observation then advances its MH state machine.  Attempts per observation
 *     double per round.
 *   - Global tail (several GPUs): an observation that needs 10^5..10^8 attempts is a
 *     millisecond of a whole GPU, and the sweep ends when the unluckiest rank does.  From
 *     K = k_switch attempts per round on, the ranks therefore gather their pending observations
 *     into every rank's exchange window (peer stores over NVLink) and search them TOGETHER:
 *     attempt block q of observation o belongs to rank (o + q) mod W, a survivor is pushed to
 *     every rank's `found` word with a system-scope atomicMin, rounds end with a flag barrier in
 *     peer memory, and every rank advances the (identical) MH state machines redundantly.  The
 *     owner replays.  No host, no NCCL call inside the sweep kernel.
 *   - Replay kernel (k_mhrs_replay, after the tail): persistent lanes stream through the record
 *     list, make the pending MH accept test, and run the accepted attempt once more with the
 *     exact FP64 walker, recording on.  A lane takes the next record as soon as its path ends
 *     (refilled eight or more lanes at a time), so the FP64-heavy recording code runs on nearly
 *     full warps -- inside the lane kernel it ran in waves at a third of the lanes and was a
 *     third of that kernel's instructions (profiles/r2c_mhrs_1e7_ncu_full.md) -- and the per-path
 *     fixed-point z goes to per-lane integer accumulators, reduced once at the end (n <= 8).
 *   - Statistics: N, B in shared-memory integer atomics; z per path in FP64 exactly like the
 *     reference's z2, then added as int64 fixed point, so the sweep totals do not depend on
 *     scheduling or on the number of GPUs.
 *
 * Roofline: issue bound (one Philox block per jump-step; 9..13 B of HBM per path).
 */
#include <cooperative_groups.h>
#include "engine_internal.h"
#include "pht_philox.h"

namespace cg = cooperative_groups;

#ifndef MHRS_THREADS
#define MHRS_THREADS 256
#endif
#define MHRS_WARPS (MHRS_THREADS / 32)
#ifndef MHRS_MIN_BLOCKS
#define MHRS_MIN_BLOCKS 4                /* lane kernel: 64 registers, 32 warps per SM */
#endif
#ifndef MHRS_TAIL_MIN_BLOCKS
#define MHRS_TAIL_MIN_BLOCKS 3           /* tail kernel: 80 registers, 24 warps per SM */
#endif
/* rare-path helpers (exact walker, replay): inlined, because a call inside the search loops makes ptxas keep the
 * loop-carried walk state in local memory (measured: 15 LDL/STL per jump-step); -DMHRS_NOINLINE_COLD to compare */
#ifndef MHRS_NOINLINE_COLD
#define MHRS_COLD static __device__ __forceinline__
#else
#define MHRS_COLD static __device__ __noinline__
#endif
#define GUIDE_BITS 8
#define GUIDE (1 << GUIDE_BITS)     /* buckets of the scan guide table */
#ifndef END_CAP
#define END_CAP 32u                 /* attempts a lane still tries once no observations are left */
#endif
#ifndef MHRS_REPLAY_MIN_BLOCKS
#define MHRS_REPLAY_MIN_BLOCKS 4         /* replay kernel: 64 registers, 32 warps per SM (measured against 3 blocks at 80: 1.27 vs 1.42 ms per sweep of 1e7) */
#endif
#ifndef REPLAY_REFILL_MIN
#define REPLAY_REFILL_MIN 16        /* idle lanes of a warp that trigger a refill from the record list */
#endif
#ifndef EV_MIN
#define EV_MIN 8u                   /* lane kernel: lanes with an event that make the warp leave the step loop ... */
#endif
#ifndef EV_WAIT
#define EV_WAIT 16u                 /* ... or steps the first of them has waited (lane kernel per sweep of 1e7, ms: 1/1 4.82, 3/4 4.58, 5/8 4.44, 8/16 4.38, 16/32 4.50) */
#endif
#ifndef PREFETCH_MIN
#define PREFETCH_MIN 8              /* empty prefetch slots in a warp that trigger a refill */
#endif
#ifndef TAIL_CH
#define TAIL_CH 256u                /* attempts per tail chunk (a pool never crosses a chunk) */
#endif
#ifndef TAIL_BATCH
#define TAIL_BATCH 1u               /* consecutive attempts a lane takes from a pool at once (measured: 1 beats 2, 4, 8) */
#endif
#ifndef TAIL_LATE_P
#define TAIL_LATE_P 1024u           /* from this few pending observations on, K grows by TAIL_LATE_GROWTH per round */
#endif
#ifndef TAIL_LATE_GROWTH
#define TAIL_LATE_GROWTH 4u
#endif
#ifndef DRAIN_LANES
#define DRAIN_LANES 32              /* END_CAP applies once this few lanes of the warp still hold an observation (32 = at once; 8 measured slower) */
#endif
#ifndef TAIL_K0
#define TAIL_K0 512u                /* attempts per pending observation in tail round 0 (a multiple of TAIL_CH) */
#endif
#define TAIL_KMAX (1u << 24)
#ifndef TAIL_GROWTH
#define TAIL_GROWTH 2u              /* K grows by this factor per round */
#endif
#ifndef FOUND_PERIOD
#define FOUND_PERIOD 8u             /* steps between looks at the pool observation's `found` word (power of two) */
#endif
#define POOL_MIN 32u
#ifndef POOL_MAX
#define POOL_MAX 256u
#endif
#define FOUND_NONE 0xFFFFFFFFFFFFFFFFull
#define T52_NEVER (1ull << 52)
#define LOWBITS (1u << 20)          /* exponential uniforms below 2^-12 go to the exact walker */
#define XBAR_TIMEOUT_NS 4000000000ull

/* record of a finished observation (SweepParams::recs[position]): x = accepted attempt so far, y = proposal, z = flags
 * (bits 8..15: end state of x, bits 16..23: end state of y) */
#define RF_PROP 2u                  /* y holds an MH proposal whose accept test is still to be made */
#define RF_OFF 4u                   /* x runs one draw into its sub-stream */
#define RF_SKIP 8u                  /* no path (the observation was dropped with error word 8) */

template <int NC>
struct MhrsSmem {
    static constexpr int R = NC + 1;            /* rows: states 0..n-1, row n = the start distribution */
    unsigned long long thr[R * R];              /* integer scan thresholds (see build_tables) */
    double cum[R * R];                          /* running sums: the exact walker's scan */
    double scale[NC];                           /* 1 / -S_jj */
    double s[NC];                               /* exit rates (MH accept ratio) */
    double inv_smax;                            /* 1 / max_j scale[j]: the filter clock's unit */
    unsigned long long zlo[NC];                 /* fixed-point sojourn totals, two limbs (engine_internal.h) */
    long long zhi[NC];
    unsigned int Nacc[NC * NC];
    unsigned int Bacc[NC];
    float A[R + 3];                             /* -ln2 * scale[k] / smax (entry n = 0: absorbed, the clock stands) */
    unsigned int paths_done;                    /* replays finished by this block */
    unsigned int scan[MHRS_WARPS + 1];          /* block-level compaction of the global list */
    uint32_t pctr[MHRS_WARPS];                  /* tail: next attempt of each warp's current pool */
    /* per-lane state that is touched once or twice per observation lives here, not in registers: the prefetched
     * next observation and the MH bookkeeping */
    float pf_yf[MHRS_THREADS]; uint32_t pf_og[MHRS_THREADS], pf_pos[MHRS_THREADS];
    uint32_t mh_cur_a[MHRS_THREADS], mh_misc[MHRS_THREADS];     /* misc: cur_pre | cur_off << 8 | kprop << 16 */
    unsigned char guide[R * GUIDE];
};

__device__ __forceinline__ unsigned long long gtimer() {
    unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t;
}
__device__ __forceinline__ float lg2_approx(float x) {
    float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r;
}

/* Philox4x32-10 block (b, a, observation, sweep) with the round keys taken from the kernel parameters */
__device__ __forceinline__ pht_u32x4 philox_block(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const SweepParams &p) {
    PHT_PHILOX_ROUND(p.rk.k[0], p.rk.k[1])   PHT_PHILOX_ROUND(p.rk.k[2], p.rk.k[3])   PHT_PHILOX_ROUND(p.rk.k[4], p.rk.k[5])
    PHT_PHILOX_ROUND(p.rk.k[6], p.rk.k[7])   PHT_PHILOX_ROUND(p.rk.k[8], p.rk.k[9])   PHT_PHILOX_ROUND(p.rk.k[10], p.rk.k[11])
    PHT_PHILOX_ROUND(p.rk.k[12], p.rk.k[13]) PHT_PHILOX_ROUND(p.rk.k[14], p.rk.k[15]) PHT_PHILOX_ROUND(p.rk.k[16], p.rk.k[17])
    PHT_PHILOX_ROUND(p.rk.k[18], p.rk.k[19])
    pht_u32x4 out; out.v[0] = c0; out.v[1] = c1; out.v[2] = c2; out.v[3] = c3;
    return out;
}

/* ------------------------------------------------------------------------------------------ exact walker
 * The chain of one attempt in the reference's arithmetic: sub-stream a, next Philox block b, time t of the
 * pending exit from state j. */
struct Walk {
    double t, spare;
    uint32_t spare_hi, a, b;
    int j;
    bool odd, fresh;
};
/* recording state of a replayed path */
struct Rec { double lastt; int B; long out_idx; double *z2; };

/* position the walk on the first draw of attempt a; off = the MH accept uniform of the previous proposal
 * occupies draw 0 of this sub-stream (src/Simulate_AbsCTMC_eq_Bladt_MHRS.c:79) */
__device__ __forceinline__ void walk_begin(Walk &w, uint32_t a, bool off, uint32_t og, const SweepParams &p, uint32_t iter) {
    w.a = a; w.fresh = true; w.b = 0; w.odd = false; w.t = 0.0; w.j = 0; w.spare = 0.0; w.spare_hi = 0u;
    if (off) {
        pht_u32x4 r = philox_block(0u, a, og, iter, p);
        w.spare = pht_u01(r.v[2], r.v[3]); w.spare_hi = r.v[3]; w.odd = true; w.b = 1;
    }
}

/* log of a uniform in (0,1): always a positive normal number, so the core of pht_log applies directly */
__device__ __forceinline__ double log_unit(double x) { return pht_log_core(pht_d2u(x), 0); }

/* One jump-step of an exact walk; returns true when the attempt ended on this step (w.t, w.j are then the exit
 * time and the state occupied at the end). */
template <bool RECORD, int NC>
__device__ __forceinline__ bool walk_step(Walk &w, double y, bool cens, uint32_t og, const SweepParams &p, MhrsSmem<NC> &sm,
                                          uint32_t iter, int n, Rec &rec) {
    constexpr int R = NC + 1;
    pht_u32x4 r = philox_block(w.b, w.a, og, iter, p);
    w.b++;
    const double f = pht_u01(r.v[0], r.v[1]), g = pht_u01(r.v[2], r.v[3]);
    const double uA = w.odd ? w.spare : f;               /* start state / next state */
    const uint32_t hiA = w.odd ? w.spare_hi : r.v[1];
    const double uB = w.odd ? f : g;                     /* next exponential */
    w.spare = g; w.spare_hi = r.v[3];
    const bool fresh = w.fresh;
    const int row = fresh ? n : w.j;
    const int last = fresh ? n - 1 : n;
    const double *c = sm.cum + row * R;
    /* reference scan `while (sofar < target) sofar += p[k++]` = number of leading running sums below the target
     * among the first `last`.  The guide entry counts the sums <= bucket floor < uA. */
    int k = sm.guide[row * GUIDE + (hiA >> (32 - GUIDE_BITS))] & 0x7f;
    while (k < last && c[k] < uA) k++;
    const bool cont = (k < n) && (w.t < y || cens);                /* gt_Bladt_MHRS.c:75,111 */
    const bool ended = !fresh && !cont;
    const bool advance = !fresh && cont;
    if (RECORD) {
        if (advance) {
            rec.z2[w.j] += w.t - rec.lastt;                                        /* :112 */
            if (p.outN != nullptr) p.outN[(size_t)rec.out_idx * n * n + w.j + k * n]++;
            else atomicAdd(&sm.Nacc[w.j + k * n], 1u);                             /* :113 */
        }
        rec.lastt = fresh ? 0.0 : (advance ? w.t : rec.lastt);
        rec.B = fresh ? k : rec.B;
    }
    const double tb = fresh ? 0.0 : w.t;
    const int jn = ended ? w.j : k;
    const double tn = tb + sm.scale[jn] * (-log_unit(uB));         /* :80, rexp(1/-S_jj) */
    w.t = ended ? w.t : tn;
    w.j = jn;
    w.fresh = false;
    return ended;
}

/* Run attempt a of observation (y, cens, og) to its end with the exact walker.  Returns true when it survives
 * (alive at y in a state that can exit, eq_Bladt_MHRS.c:66,74); *jend = the state it is in at the end.
 * IV: an interval-censored observation (cens with u < inf) survives only when it is absorbed at t <= u as well. */
/* result word: bit 0 survived, bits 8..15 end state, bits 16..31 jump-steps taken */
template <int NC, bool IV = false>
MHRS_COLD uint32_t exact_attempt(uint32_t a, bool off, double y, bool cens, uint32_t og, const SweepParams &p,
                                                      MhrsSmem<NC> &sm, uint32_t iter, int n, uint32_t smask, double u = 0.0) {
    Walk w; Rec norec; norec.lastt = 0.0; norec.B = 0; norec.out_idx = 0; norec.z2 = nullptr;
    walk_begin(w, a, off, og, p, iter);
    unsigned st = 1;
    while (!walk_step<false>(w, y, cens, og, p, sm, iter, n, norec)) st++;
    bool ok = (w.t >= y) && ((smask >> w.j) & 1u);
    if constexpr (IV) ok = ok && w.t <= u;
    return (ok ? 1u : 0u) | ((uint32_t)w.j << 8) | ((st > 0xffffu ? 0xffffu : st) << 16);
}

/* ------------------------------------------------------------------------------------------ replay
 * Persistent lanes over the record list [obs_begin, obs_end): gt_Bladt_MHRS.c:135-137, then eq_Bladt_MHRS.c:79-82 (the
 * accept test left pending by the lane phase when mhit = 1) and :104-110.  Finished lanes park until REPLAY_REFILL_MIN of
 * the warp are idle (or nothing is left), then fold their path into the statistics and take new records together. */
template <int NC>
__device__ __forceinline__ void replay_phase(const SweepParams &p, MhrsSmem<NC> &sm, uint32_t iter, int n,
                                             uint32_t obs_begin, uint32_t obs_end, unsigned &c_jumps) {
    const unsigned FULL = 0xffffffffu; const int lane = threadIdx.x & 31;
    constexpr bool LANE_Z = NC <= 8;                    /* per-lane fixed-point totals in registers */
    long long ztot[LANE_Z ? NC : 1];
#pragma unroll
    for (int i = 0; i < (LANE_Z ? NC : 1); i++) ztot[i] = 0;
    double z2[NC];
    Walk w; Rec rec; rec.lastt = 0.0; rec.B = 0; rec.z2 = z2; rec.out_idx = 0;
    w.t = 0.0; w.spare = 0.0; w.spare_hi = 0u; w.a = 0u; w.b = 0u; w.j = 0; w.odd = false; w.fresh = true;
    double y = 0.0; bool cens = false, act = false, fin = false, dry = false, bad = false; uint32_t og = 0u;
    unsigned paths = 0;
    const double zs = pht_u2d((uint64_t)(1023 + p.zbits) << 52);
    for (;;) {
        const unsigned idle = __ballot_sync(FULL, !act);
        if (idle == FULL || (unsigned)__popc(idle) >= REPLAY_REFILL_MIN) {
            if (fin) {
                /* ---- the path that ended on this lane: last sojourn, exit count, start count, z in fixed point */
                fin = false; paths++;
                z2[w.j] += (cens ? w.t : y) - rec.lastt;
                if (p.outB != nullptr) {
                    p.outB[rec.out_idx] = rec.B;
                    p.outN[rec.out_idx * n * n + w.j + w.j * n]++;
#pragma unroll 1
                    for (int i = 0; i < n; i++) p.outz[rec.out_idx * n + i] = z2[i];
                } else {
                    atomicAdd(&sm.Nacc[w.j + w.j * n], 1u); atomicAdd(&sm.Bacc[rec.B], 1u);
#pragma unroll
                    for (int i = 0; i < NC; i++) {
                        if (i < n) {
                            const double v = z2[i];
                            bad = bad || !(v * zs < 4.0e18);
                            const long long fx = __double2ll_rn(v * zs);
                            if (LANE_Z) { ztot[LANE_Z ? i : 0] += fx; bad = bad || ztot[LANE_Z ? i : 0] < 0; }
                            else if (fx != 0) pht_zfix_add(sm.zlo, sm.zhi, i, fx);
                        }
                    }
                }
            }
            if (!dry) {
                const unsigned cnt = __popc(idle);
                unsigned long long base = 0;
                if (lane == 0) base = (unsigned long long)obs_begin + atomicAdd(&p.state->replay_next, (unsigned long long)cnt);
                base = __shfl_sync(FULL, base, 0);
                const unsigned long long left = base < obs_end ? (unsigned long long)obs_end - base : 0ull;
                const unsigned avail = left < cnt ? (unsigned)left : cnt;
                if (avail < cnt) dry = true;
                const unsigned rank = __popc(idle & ((1u << lane) - 1u));
                if (!act && rank < avail) {
                    const unsigned long long pos = base + rank;
                    const uint4 r = p.recs[pos];
                    if (!(r.z & RF_SKIP)) {
                        const uint32_t obs_local = p.perm ? p.perm[pos] : (uint32_t)pos;
                        y = p.y[pos]; cens = p.cens[pos] != 0; og = p.obs_rank + obs_local * p.obs_world;
                        rec.out_idx = (long)obs_local - p.first; rec.lastt = 0.0; rec.B = 0;
                        uint32_t a = r.x;
                        if (r.z & RF_PROP) {                                                   /* eq_Bladt_MHRS.c:79-82 */
                            const pht_u32x4 q = philox_block(0u, r.y + 1u, og, iter, p);
                            const double U = pht_u01(q.v[0], q.v[1]);
                            if (U < sm.s[(r.z >> 16) & 0xffu] / sm.s[(r.z >> 8) & 0xffu]) a = r.y;
                        }
#pragma unroll
                        for (int i = 0; i < NC; i++) z2[i] = 0.0;
                        walk_begin(w, a, (r.z & RF_OFF) != 0u, og, p, iter);
                        act = true;
                    }
                }
            }
        }
        if (__ballot_sync(FULL, act) == 0u) { if (dry) break; else continue; }
        __syncwarp();
        if (act) { c_jumps++; if (walk_step<true>(w, y, cens, og, p, sm, iter, n, rec)) { act = false; fin = true; } }
    }
    /* (the loop ends through the refill branch with every lane idle: nothing is left parked) */
    if (p.outB == nullptr) {
        if (LANE_Z) {
#pragma unroll
            for (int i = 0; i < NC; i++) {
                if (i < n) {
                    const long long fx = ztot[LANE_Z ? i : 0];
                    unsigned long long lo = (unsigned long long)fx & 0xffffffffull; long long hi = fx >> 32;
                    for (int d = 16; d > 0; d >>= 1) { lo += __shfl_xor_sync(FULL, lo, d); hi += __shfl_xor_sync(FULL, hi, d); }
                    if (lane == 0 && (lo | (unsigned long long)hi)) {
                        atomicAdd(&sm.zlo[i], lo); atomicAdd(reinterpret_cast<unsigned long long *>(&sm.zhi[i]), (unsigned long long)hi);
                    }
                }
            }
        }
        if (bad) atomicOr(&p.state->error, 2);
    }
    for (int d = 16; d > 0; d >>= 1) paths += __shfl_xor_sync(FULL, paths, d);
    if (lane == 0 && paths) atomicAdd(&sm.paths_done, paths);
}

/* ------------------------------------------------------------------------------------------ filter walk
 * What a search needs to know of its observation: y in FP32 in units of the largest mean sojourn (smax = max_j
 * scale[j]; the filter clock runs in those units so that its error constants are pure numbers), the part c0y of the
 * per-step error bound that depends on y (so that a step need not take it from y again), the Philox word, and the
 * censoring flag. */
struct ObsF { float yn, c0y; uint32_t og; bool cens; };
__device__ __forceinline__ float bound_c0(float bn) { return __fmaf_rn(1.2e-7f, bn, 4.5e-7f); }
__device__ __forceinline__ void obs_set(ObsF &o, float yn, uint32_t og, bool cens) { o.yn = yn; o.c0y = bound_c0(yn); o.og = og; o.cens = cens; }
/* IV instance: also the upper bound u in the same units (+inf: none).  c0y is then taken at the largest clock value a
 * decision is made at (u when finite, else y). */
struct ObsFU : ObsF { float un; };
template <bool IV> struct ObsOf { typedef ObsF T; };
template <> struct ObsOf<true> { typedef ObsFU T; };
__device__ __forceinline__ void obs_set_u(ObsF &, float) {}
__device__ __forceinline__ void obs_set_u(ObsFU &o, float un) { o.un = un; o.c0y = bound_c0((un < __int_as_float(0x7f800000)) ? un : o.yn); }
/* the bound of the observation at layout position pos (IV), or nothing */
template <bool IV> __device__ __forceinline__ double upper_at(const double *u, uint32_t pos) {
    if constexpr (IV) return u[pos]; else return 0.0;
}
/* the filter walk of one attempt: FP32 clock t with error bound dacc, sub-stream a, next block b, scan row */
struct Fast { float t, dacc; uint32_t a, b; int row; };

__device__ __forceinline__ void fast_begin(Fast &f, uint32_t a, int n) { f.t = 0.0f; f.dacc = 0.0f; f.a = a; f.b = 0u; f.row = n; }

/* One jump-step of the filter walk.
 * The next state is exact: with x the 52 random bits of the state uniform u = (x + 0.5) 2^-52, `cum[k] < u` <=>
 * x >= thr[k] (build_tables), and rows end with a NEVER entry so the scan needs no bound check.
 * The clock advances by (scale[k] / smax) * -ln(u) in FP32, with u taken from the top 32 bits w of the exponential
 * uniform: w -> FP32 (I2F), exponent and mantissa split, lg2.approx of the mantissa in [1, 2) (documented absolute
 * error 2^-22 there), L = (exponent - 32) + lg2(mantissa), t = fma(L, A[k], t) with A[k] = -ln2 scale[k] / smax.
 * Error of one step, in clock units (scale[k] / smax <= 1):
 *     truncation of u to w           relative 1/w <= 2^-(exponent)          -> |d ln u| <= 2^-e     (`trunc`)
 *     I2F rounding                   relative 2^-24                         -> 6.0e-8
 *     lg2.approx of the mantissa     absolute 2^-22 in log2                 -> 1.65e-7
 *     rounding of L, of A[k]         relative 2^-24 each, times ln2 |L|     -> 8.3e-8 |L|
 *     rounding of the FMA            relative 2^-24 of t_new <= y + ln2 |L| -> 6.0e-8 y + 4.1e-8 |L|
 * (a clock beyond 2y is in no danger: its relative error stays below 1e-3 for the 4096 steps a walk may take here.)
 * The bound accumulated per step is TWICE that sum: 2 * 2^-e + (4.5e-7 + 1.2e-7 y) + 2.5e-7 |L|.  Uniforms with
 * w < 4096 and walks of 4096 steps make the bound infinite, i.e. leave the decision to the exact walker.
 * Outcome of the step: fail (the attempt is dead for certain), surv (alive at y for certain, in state f.row), amb (the
 * clock is inside the error band at the moment of the test: ask the exact walker), none of them (the walk goes on).
 * IV (interval-censored observations, absorbed in [y, u]): the same bound, with its clock-proportional part taken at u
 * instead of y, gives a second band around u.  The attempt fails as soon as the clock is past u for certain (the clock
 * only grows), survives when absorbed above y and below u for certain, and goes to the exact walker inside either band.
 *
 * Almost every step has none of these outcomes, so the step only works out whether the attempt ENDS here and whether
 * it failed; fast_survives tells surv from amb afterwards, for the attempts that ended without failing.  The step at
 * which `alive at y` is decided is absorption for a censored observation and any other step for an exact one, so an
 * attempt ends at absorption, at a step of an exact observation not dead at y for certain, or (IV) past u for certain.
 * It fails when absorbed before y (exact) or dead at y for certain (censored), or (IV) past u.  Because `over` and
 * `under` (and `past` and `below`) exclude each other, the outcomes are those of the test above.
 * c0y = the part of the bound that depends on y (ObsF).  On absorption f.row keeps the state the chain was absorbed
 * from: the state occupied at the end. */
template <int NC, bool IV = false>
__device__ __forceinline__ bool fast_step(Fast &f, const typename ObsOf<IV>::T &o, float c0y, const SweepParams &p, const MhrsSmem<NC> &sm,
                                          uint32_t iter, int n, bool &fail) {
    constexpr int R = NC + 1;
    const pht_u32x4 r = philox_block(f.b, f.a, o.og, iter, p);
    f.b++;
    const unsigned g = sm.guide[f.row * GUIDE + (r.v[1] >> (32 - GUIDE_BITS))];
    int k = (int)(g & 0x7fu);
    /* bit 7: no threshold of the row falls inside the bucket, the guide entry IS the answer (24 of 25 look-ups at 8
     * phases); only the other buckets need the 52 bits x */
    if (!(g & 0x80u)) {
        const unsigned long long x = (((unsigned long long)r.v[1] << 32) | r.v[0]) >> 12;
        const unsigned long long *th = sm.thr + f.row * R;
        while (x >= th[k]) k++;
    }
    const uint32_t w = r.v[3];
    const uint32_t wb = __float_as_uint(__uint2float_rn(w));
    const uint32_t eb = wb >> 23;                                                     /* 127 + exponent of w */
    const float lg2m = lg2_approx(__uint_as_float((wb & 0x007fffffu) | 0x3f800000u));
    const float L = (__uint_as_float(0x4b400000u + eb) - 12583071.0f) + lg2m;        /* (eb - 159) + lg2m: log2 of u */
    f.t = __fmaf_rn(L, sm.A[k], f.t);
    const float trunc = __uint_as_float((254u - eb) << 23);                           /* 2^-(exponent of w) >= 1 / w */
    const float step_err = __fmaf_rn(trunc, 2.0f, __fmaf_rn(fabsf(L), 2.5e-7f, c0y));
    const bool flagged = (w < 4096u) || (f.b >> 12) != 0u;
    f.dacc = flagged ? __int_as_float(0x7f800000) : f.dacc + step_err;
    const bool absd = (k == n);
    const bool under = -(f.t - o.yn) > f.dacc;                    /* dead at y for certain */
    bool end = absd || (!o.cens && !under);
    fail = absd && (!o.cens || under);
    if constexpr (IV) {
        const bool past = f.t - o.un > f.dacc;                  /* above u for certain */
        end = end || past;
        fail = fail || past;
    }
    f.row = absd ? f.row : k;
    return end;
}

/* after a step that ended the attempt without failing: alive at y for certain (and, IV, absorbed below u for certain);
 * otherwise the step was ambiguous */
template <bool IV>
__device__ __forceinline__ bool fast_survives(const Fast &f, const typename ObsOf<IV>::T &o) {
    bool s = f.t - o.yn > f.dacc;
    if constexpr (IV) s = s && -(f.t - o.un) > f.dacc;
    return s;
}

/* Scan tables of the sweep's model.  thr[row][k] = the smallest x in [0, 2^52] whose uniform (x + 0.5) 2^-52
 * exceeds cum[row][k] (NEVER = 2^52 when none does, also for NaN sums, and for every k beyond the row's last
 * category).  guide[row][b] = number of leading sums <= b / GUIDE: every uniform of bucket b is above them. */
template <int NC>
__device__ __forceinline__ void build_tables(const SweepParams &p, MhrsSmem<NC> &sm, int n, const ModelLayout &ML) {
    constexpr int R = NC + 1;
    const int tid = threadIdx.x;
    double smax = 0.0;
    for (int i = 0; i < n; i++) { const double sc = p.model[ML.scale + i]; smax = (sc > smax) ? sc : smax; }
    const double inv_smax = 1.0 / smax;          /* smax = 0 or NaN: the clock is NaN, every decision goes to the exact walker */
    for (int i = tid; i < n; i += MHRS_THREADS) {
        const double sc = p.model[ML.scale + i];
        sm.scale[i] = sc; sm.s[i] = p.model[ML.s + i]; sm.zlo[i] = 0ull; sm.zhi[i] = 0; sm.Bacc[i] = 0u;
        sm.A[i] = (float)((-0.69314718055994530942 * sc) * inv_smax);
    }
    if (tid == 0) { sm.A[n] = 0.0f; sm.inv_smax = inv_smax; }
    for (int i = tid; i < n * n; i += MHRS_THREADS) sm.Nacc[i] = 0u;
    for (int e = tid; e < R * R; e += MHRS_THREADS) {
        const int row = e / R, k = e % R;
        unsigned long long t52 = T52_NEVER; double c = 0.0;
        if (row <= n && k <= n) {
            c = p.model[ML.cum + row * (n + 1) + k];
            const int last = (row == n) ? n - 1 : n;
            if (k < last && c < 1.0) {                   /* NaN compares false: NEVER */
                if (!(c > 0.0)) t52 = 0ull;
                else {
                    /* floor(c 2^52) is exact; the answer is that or the next integer */
                    const unsigned long long xf = (unsigned long long)(c * 4503599627370496.0);
                    const double u = pht_u2d(0x3ff0000000000000ULL | xf) - 0.99999999999999988898;
                    t52 = (u > c) ? xf : xf + 1ull;
                }
            }
        }
        sm.thr[e] = t52; sm.cum[e] = c;
    }
    if (tid == 0) sm.paths_done = 0u;
    __syncthreads();
    for (int e = tid; e < (n + 1) * GUIDE; e += MHRS_THREADS) {
        const int row = e / GUIDE, b = e % GUIDE, last = (row == n) ? n - 1 : n;
        const double floor_u = (double)b * (1.0 / GUIDE);
        int k = 0;
        while (k < last && sm.cum[row * R + k] <= floor_u) k++;
        /* bit 7: every x of the bucket, [b, b + 1) 2^(52 - GUIDE_BITS), is below the next threshold */
        const bool pure = sm.thr[row * R + k] >= ((unsigned long long)(b + 1) << (52 - GUIDE_BITS));
        sm.guide[e] = (unsigned char)(k | (pure ? 0x80 : 0));
    }
    __syncthreads();
}

__device__ __forceinline__ uint32_t pack_flags(bool have_cur, bool cur_off, bool off, bool cens, int cur_pre, uint32_t kprop) {
    return (have_cur ? TI_HAVE : 0u) | (cur_off ? TI_CUROFF : 0u) | (off ? TI_OFF : 0u) | (cens ? TI_CENS : 0u) |
           ((uint32_t)(cur_pre & 0xff) << 8) | (kprop << 16);
}

/* barrier over the ranks of the run through the exchange windows: every thread's peer stores are fenced, the grid
 * meets, rank flags are exchanged, the grid meets again.  Gives up (error word 64) when a peer does not arrive. */
__device__ __forceinline__ void peer_barrier(cg::grid_group &grid, const SweepParams &p, unsigned long long epoch) {
    const unsigned long long t_in = (blockIdx.x == 0 && threadIdx.x == 0) ? gtimer() : 0ull;
    __threadfence_system();
    grid.sync();
    if (blockIdx.x == 0) {
        const int t = threadIdx.x;
        if (t < (int)p.obs_world && p.state->xdead == 0u) {
            volatile unsigned long long *mine = &p.xpeer[t]->flags[p.obs_rank];
            __threadfence_system();
            *mine = epoch;
            __threadfence_system();
            volatile unsigned long long *theirs = &p.xw->flags[t];
            const unsigned long long t0 = gtimer();
            while (*theirs < epoch) {
                if (gtimer() - t0 > XBAR_TIMEOUT_NS) { p.state->xdead = 1u; atomicOr(&p.state->error, 64); break; }
            }
            __threadfence_system();
        }
    }
    grid.sync();
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&p.state->counters[PHT_CNT_NS_XWAIT], gtimer() - t_in);
}

/* ------------------------------------------------------------------------------------------ tail search
 * One round: K attempts for each of the P pending observations.  Units are numbered chunk-major: local chunk c
 * covers attempt block q = c / Pl of the observation in column i = c % Pl, so every observation's first chunk is
 * handed out before any second chunk, and later chunks are mostly skipped once an earlier one has survived.
 * Local rounds: Pl = P, column i is pend[i].  Global rounds (W ranks): Pl = ceil(P / W), column i of block q is
 * observation i W + (rank - q) mod W, i.e. block q of observation o is searched by rank (o + q) mod W. */
struct TailView {
    TailItem *items; const uint32_t *pend; unsigned long long *found; uint32_t P, K;
    bool global; uint32_t parity;
    const double *u;           /* IV: the items' upper bounds, indexed like items */
};

template <int NC, bool IV = false>
__device__ __forceinline__ void tail_search(const TailView &tv, const SweepParams &p, MhrsSmem<NC> &sm, uint32_t iter, int n,
                                            uint32_t smask, uint32_t nwarps,
                                            unsigned &c_jumps, unsigned &c_attempts) {
    const unsigned FULL = 0xffffffffu; const int lane = threadIdx.x & 31;
    const uint32_t W = tv.global ? p.obs_world : 1u;
    const uint32_t Pl = (tv.P + W - 1u) / W;
    const unsigned long long total_units = (unsigned long long)Pl * tv.K;
    /* per lane: the attempt f.a of observation my_item it is walking.  Attempts are handed out ONE at a time from the
     * warp's current pool through a counter in shared memory: a lane whose attempt has failed takes the next one inside
     * its own branch (one ATOMS), so the warp-wide hand-out code -- which with whole-warp ballots ran on almost every
     * iteration, some lane fails in most of them -- is left for the moment a pool runs out. */
    Fast f; fast_begin(f, 0u, n);
    typename ObsOf<IV>::T mo; obs_set(mo, 0.0f, 0u, false); obs_set_u(mo, 0.0f);
    uint32_t my_item = 0xFFFFFFFFu; bool active = false;
    unsigned steps = 0;
    uint32_t *ctr = &sm.pctr[threadIdx.x >> 5];
    if (lane == 0) *ctr = 0u;
    __syncwarp();
    /* warp-uniform: the units this warp holds, and the pool being handed out ([*ctr, pool_end) of observation `item`) */
    unsigned long long u_next = 0, u_end = 0, last_base = 0, remaining = total_units;
    bool out_of_units = false, finished = false;
    uint32_t item = 0, og = 0, a_first = 0, pool_end = 0; float yf = 0.0f, uf = 0.0f; bool cens = false, first_off = false;
    while (!finished) {
        /* ---- the search loop proper: no calls in here (the exact walker is asked from outside, see below) */
        bool want_exact = false, exact_off = false, survived = false; int kend = 0;
        /* take the pool's next attempt (any lane, any time) */
#define TAIL_GRAB() do { \
            const uint32_t na_ = atomicAdd(ctr, 1u); \
            if (na_ < pool_end) { \
                my_item = item; obs_set(mo, yf, og, cens); obs_set_u(mo, uf); fast_begin(f, na_, n); \
                /* the attempt that starts one draw into its sub-stream (after an MH accept test) is the exact walker's */ \
                if (first_off && na_ == a_first) { want_exact = true; exact_off = true; active = false; } else active = true; \
            } else active = false; \
        } while (0)
        for (;;) {
            const unsigned idle = __ballot_sync(FULL, !active);
            if (idle) {
                uint32_t cur = *reinterpret_cast<volatile uint32_t *>(ctr);
                if (cur >= pool_end && !out_of_units) {
                    /* take the next pool (skipping pools that an earlier survivor made moot) */
                    bool have = false; uint32_t pstart = 0u;
                    while (!have) {
                        if (u_next >= u_end) {
                            remaining = total_units > last_base ? total_units - last_base : 0ull;
                            unsigned long long want = remaining / (2ull * (unsigned long long)nwarps);
                            want = want < POOL_MIN ? POOL_MIN : (want > POOL_MAX ? POOL_MAX : want);
                            unsigned long long base = 0;
                            if (lane == 0) base = atomicAdd(&p.state->unit_counter, want);
                            base = __shfl_sync(FULL, base, 0);
                            last_base = base;
                            if (base >= total_units) { out_of_units = true; break; }
                            u_next = base; u_end = base + want < total_units ? base + want : total_units;
                        }
                        const unsigned long long chunk = u_next / TAIL_CH;
                        const unsigned long long chunk_end_u = (chunk + 1ull) * TAIL_CH;
                        const unsigned long long stop = u_end < chunk_end_u ? u_end : chunk_end_u;
                        const uint32_t q = (uint32_t)(chunk / Pl), col = (uint32_t)(chunk % Pl);
                        const uint32_t o = tv.global ? col * W + (p.obs_rank + W - q % W) % W : col;
                        const uint32_t within = (uint32_t)(u_next - chunk * TAIL_CH), len = (uint32_t)(stop - u_next);
                        u_next = stop;
                        if (o >= tv.P) continue;
                        const uint32_t it_idx = tv.pend[o];
                        const TailItem it = tv.items[it_idx];
                        if (it.flags & TI_FIN) continue;
                        pstart = it.a + q * TAIL_CH + within;
                        if ((__ldcg(&tv.found[it_idx]) >> 8) >= (unsigned long long)pstart) {
                            have = true;
                            item = it_idx; a_first = it.a; first_off = (it.flags & TI_OFF) != 0u;
                            pool_end = pstart + len;
                            yf = (float)(it.y * sm.inv_smax); cens = (it.flags & TI_CENS) != 0u; og = it.og;
                            if constexpr (IV) uf = (float)(tv.u[it_idx] * sm.inv_smax);
                        }
                    }
                    if (have) {
                        __syncwarp();
                        if (lane == 0) *ctr = pstart;
                        __syncwarp();
                        cur = pstart;
                    }
                }
                if (cur >= pool_end) { if (idle == FULL) { finished = true; break; } }      /* nothing in flight, nothing left to hand out */
                else if (!active) TAIL_GRAB();
            }
            /* Every FOUND_PERIOD steps, look whether someone (another warp, another GPU) has found a surviving attempt
             * of the pool's observation: everything above it is moot. */
            if (((++steps) & (FOUND_PERIOD - 1u)) == 0u) {
                unsigned long long fw = 0;
                if (lane == 0) fw = __ldcg(&tv.found[item]);
                fw = __shfl_sync(FULL, fw, 0);
                if (fw != FOUND_NONE) {
                    const uint32_t fa = (uint32_t)(fw >> 8);
                    pool_end = pool_end < fa ? pool_end : fa;
                    if (my_item == item && active && f.a > fa) { active = false; c_jumps += f.b; }
                }
            }
            __syncwarp();           /* lanes that have just taken an attempt step together with the rest */
            if (active) {
                bool fail;
                /* (at its 80 registers the tail would spill c0y of an exact or right-censored observation: it is taken from y
                 * in each step instead; the IV instance holds it in place of the bound it is taken at) */
                if (fast_step<NC, IV>(f, mo, IV ? mo.c0y : bound_c0(mo.yn), p, sm, iter, n, fail)) {
                    const bool surv = !fail && fast_survives<IV>(f, mo);
                    if (surv && !((smask >> f.row) & 1u)) fail = true;     /* alive at y in a state that cannot exit: failed */
                    /* (jump-steps are counted when an attempt ends: f.b of them) */
                    if (fail) { c_attempts++; c_jumps += f.b; TAIL_GRAB(); }
                    else if (surv) { c_attempts++; c_jumps += f.b; survived = true; kend = f.row; active = false; }
                    else { c_jumps += f.b; want_exact = true; active = false; }
                }
            }
            if (__any_sync(FULL, survived || want_exact)) break;
        }
#undef TAIL_GRAB
        if (finished) break;
        /* ---- attempts the filter could not decide (or that start off the block boundary): the exact walker */
        if (want_exact) {
            const uint32_t res = exact_attempt<NC, IV>(f.a, exact_off, tv.items[my_item].y, mo.cens, mo.og, p, sm, iter, n, smask,
                                                       upper_at<IV>(tv.u, my_item));
            c_jumps += res >> 16; c_attempts++;
            survived = res & 1u; kend = (int)((res >> 8) & 0xffu);
        }
        /* ---- every survivor competes for "lowest surviving attempt" of its observation (on every rank in a global
         * round); the first one in the warp also calls off the later attempts of the same observation in flight here */
        const unsigned smk = __ballot_sync(FULL, survived);
        if (survived) {
            const unsigned long long word = ((unsigned long long)f.a << 8) | (unsigned long long)kend;
            atomicMin(&tv.found[my_item], word);
            if (tv.global) {
                for (uint32_t r = 0; r < p.obs_world; r++)
                    if (r != p.obs_rank) atomicMin_system(&p.xpeer[r]->gfound[tv.parity][my_item], word);
                __threadfence_system();
            }
        }
        if (smk) {
            const int src = __ffs(smk) - 1;
            const uint32_t s_item = __shfl_sync(FULL, my_item, src), s_a = __shfl_sync(FULL, f.a, src);
            if (my_item == s_item && active && f.a > s_a) { active = false; c_jumps += f.b; }
            if (s_item == item) pool_end = pool_end < s_a ? pool_end : s_a;
        }
        __syncwarp();
    }
}

/* advance one pending observation's MH state machine after a round (eq_Bladt_MHRS.c:65-101); returns 0 = still
 * pending, 1 = finished (accepted attempt known), 2 = dropped */
MHRS_COLD int tail_advance(TailItem &it, unsigned long long fword, uint32_t K, const SweepParams &p,
                                            const double *s_model, uint32_t iter, bool &failed) {
    failed = false;
    if (fword == FOUND_NONE) {
        failed = true;
        if (it.a > 0xF0000000u - K) return 2;              /* survival probability ~ 0: see DESIGN.md */
        it.a += K; it.flags &= ~TI_OFF;
        return 0;
    }
    const uint32_t a = (uint32_t)(fword >> 8); const int pre = (int)(fword & 0xffull);
    const bool off = (a == it.a) && (it.flags & TI_OFF);
    const bool cens = (it.flags & TI_CENS) != 0u;
    bool have_cur = it.flags & TI_HAVE; bool cur_off = it.flags & TI_CUROFF;
    int cur_pre = (int)((it.flags >> 8) & 0xffu); uint32_t kprop = it.flags >> 16;
    bool next_off = false, done;
    if (!have_cur) {
        have_cur = true; it.cur_a = a; cur_off = off; cur_pre = pre;
        done = cens || p.mhit == 0;
    } else {
        pht_u32x4 r = philox_block(0u, a + 1u, it.og, iter, p);
        const double U = pht_u01(r.v[0], r.v[1]);
        if (U < s_model[pre] / s_model[cur_pre]) { it.cur_a = a; cur_off = off; cur_pre = pre; }
        kprop++; done = (int)kprop >= p.mhit; next_off = true;
    }
    it.a = a + 1u;
    it.flags = pack_flags(have_cur, cur_off, next_off, cens, cur_pre, kprop);
    return done ? 1 : 0;
}

/* ------------------------------------------------------------------------------------------ lane phase
 * Persistent warps, one observation per lane, in layout order from a global counter. */
#define LF_RUN 1u        /* the lane holds an observation and walks */
#define LF_HAVE 2u       /* a first surviving attempt is known (mh_cur_a / mh_misc) */
#define LF_CENS 4u
#define LF_NVALID 8u     /* the prefetch slot holds an observation */
#define LF_NCENS 16u
template <int NC, bool IV = false>
__device__ __forceinline__ void lane_phase(const SweepParams &p, MhrsSmem<NC> &sm, uint32_t iter, int n, uint32_t smask,
                                           uint32_t obs_begin, uint32_t obs_end, uint32_t cap,
                                           unsigned &c_jumps, unsigned &c_attempts) {
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31;
    Fast f; fast_begin(f, 0u, n);
    typename ObsOf<IV>::T o; obs_set(o, 0.0f, 0u, false); obs_set_u(o, 0.0f);
    const double inv_smax = sm.inv_smax;
    uint32_t pos = 0, a_lim = cap, fl = 0u;
    bool dry = false;                     /* warp-uniform: the observation stream has run out */
    for (;;) {
        /* ---- refill the prefetch slots, eight or more at a time */
        const unsigned empty = __ballot_sync(FULL, !(fl & LF_NVALID));
        if (!dry && __popc(empty) >= PREFETCH_MIN) {
            const unsigned cnt = __popc(empty);
            unsigned long long base = 0;
            if (lane == 0) base = (unsigned long long)obs_begin + atomicAdd(&p.state->next_obs, (unsigned long long)cnt);
            base = __shfl_sync(FULL, base, 0);
            const unsigned long long left = base < obs_end ? (unsigned long long)obs_end - base : 0ull;
            const unsigned avail = left < cnt ? (unsigned)left : cnt;
            if (avail < cnt) dry = true;
            const unsigned rank = __popc(empty & ((1u << lane) - 1u));
            if (!(fl & LF_NVALID) && rank < avail) {
                const unsigned long long q = base + rank;
                sm.pf_pos[tid] = (uint32_t)q; sm.pf_yf[tid] = (float)(p.y[q] * inv_smax);
                sm.pf_og[tid] = p.obs_rank + (p.perm ? p.perm[q] : (uint32_t)q) * p.obs_world;
                fl |= LF_NVALID | (p.cens[q] != 0 ? LF_NCENS : 0u);
            }
        }
        if (!(fl & LF_RUN) && (fl & LF_NVALID)) {
            obs_set(o, sm.pf_yf[tid], sm.pf_og[tid], (fl & LF_NCENS) != 0u); pos = sm.pf_pos[tid];
            if constexpr (IV) obs_set_u(o, (float)(p.u[pos] * inv_smax));
            fl = LF_RUN | (o.cens ? LF_CENS : 0u);
            sm.mh_cur_a[tid] = 0u; sm.mh_misc[tid] = 0u; a_lim = cap;
            fast_begin(f, 0u, n);
        }
        const unsigned running = __ballot_sync(FULL, fl & LF_RUN);
        if (running == 0u) { if (dry) break; else continue; }
        /* a few last lanes must not hold the grid: once the stream is dry and the warp is mostly idle, the rest goes
         * to the tail after END_CAP attempts */
        if (dry && __popc(running) <= DRAIN_LANES && a_lim != 0xFFFFFFFFu && a_lim > END_CAP) a_lim = END_CAP;
        __syncwarp();
        /* ---- the search loop proper: steps until some lane has something to report.  No calls, nothing but the
         * filter walk, in here; a failed attempt restarts on the next sub-stream on the spot. */
        bool go = (fl & LF_RUN) != 0u;
        /* A lane that has something to report stops walking, but the warp only leaves the loop for the (divergent, ~100
         * instructions at 2 lanes) event code once EV_MIN lanes are waiting or the first of them has waited EV_WAIT steps:
         * events come every ~150 steps per lane, so the wait costs a lane a few per cent and the event code runs a third as often.
         * Two jump-steps per vote: a lane that stops in the first sits out the second, and the vote, its count and the
         * wait counter (kept in steps) cost half as much per step.  A lane stops when its attempt ended without failing,
         * or when it failed and the next attempt is the tail's (f.b = 0 then: the walk has restarted). */
        unsigned waited = 0u, ev;
        do {
#pragma unroll
            for (int h = 0; h < 2; h++) {
                if (go) {
                    bool fail;
                    const bool end = fast_step<NC, IV>(f, o, o.c0y, p, sm, iter, n, fail);
                    if (fail) { c_jumps += f.b; fast_begin(f, f.a + 1u, n); c_attempts++; }
                    go = fail ? f.a < a_lim : !end;
                }
            }
            ev = __ballot_sync(FULL, !go);
            waited += ((ev & running) != 0u) ? 2u : 0u;
        } while (ev != 0xffffffffu && (unsigned)__popc(ev & running) < EV_MIN && waited < EV_WAIT);
        /* ---- events, a few lanes at a time */
        const bool stopped = (fl & LF_RUN) && !go;
        bool hand = stopped && f.b == 0u, surv = false, amb = false; int k = f.row;
        if (stopped && f.b != 0u) {
            c_jumps += f.b;                         /* the filter steps of the attempt that just ended (failed ones: above) */
            surv = fast_survives<IV>(f, o); amb = !surv;
        }
        if (amb) {
            const uint32_t res = exact_attempt<NC, IV>(f.a, false, p.y[pos], o.cens, o.og, p, sm, iter, n, ~0u, upper_at<IV>(p.u, pos));
            surv = res & 1u; k = (int)((res >> 8) & 0xffu); c_jumps += res >> 16;
            if (!surv) { fast_begin(f, f.a + 1u, n); c_attempts++; hand = f.a >= a_lim; }
        }
        /* survived to y in a state that cannot exit: a failed attempt (eq_Bladt_MHRS.c:66,74) */
        if (surv && !((smask >> k) & 1u)) { surv = false; fast_begin(f, f.a + 1u, n); c_attempts++; hand = f.a >= a_lim; }
        bool this_off = false;
        while (surv) {
            c_attempts++;
            bool complete = false; uint32_t rfl = 0u, ra1 = 0u, ra2 = 0u;
            uint32_t cur_a = sm.mh_cur_a[tid], misc = sm.mh_misc[tid];
            int cur_pre = (int)(misc & 0xffu); bool cur_off = (misc >> 8) & 1u; uint32_t kprop = misc >> 16;
            if (!(fl & LF_HAVE)) {
                fl |= LF_HAVE; cur_a = f.a; cur_off = this_off; cur_pre = k;
                if (o.cens || p.mhit == 0) { complete = true; ra1 = cur_a; rfl = cur_off ? RF_OFF : 0u; }        /* :70 */
            } else if (p.mhit == 1) {
                /* the one proposal: its accept test is left to the replay session (whole warp at once) */
                complete = true; ra1 = cur_a; ra2 = f.a;
                rfl = RF_PROP | ((uint32_t)cur_pre << 8) | ((uint32_t)k << 16);
            } else {
                /* a valid proposal: accept test with draw 0 of the next sub-stream (:79-82) */
                pht_u32x4 r = philox_block(0u, f.a + 1u, o.og, iter, p);
                const double U = pht_u01(r.v[0], r.v[1]);
                if (U < sm.s[k] / sm.s[cur_pre]) { cur_a = f.a; cur_off = this_off; cur_pre = k; }
                kprop++;
                if ((int)kprop >= p.mhit) { complete = true; ra1 = cur_a; rfl = cur_off ? RF_OFF : 0u; }
            }
            sm.mh_cur_a[tid] = cur_a; sm.mh_misc[tid] = (uint32_t)cur_pre | (cur_off ? 0x100u : 0u) | (kprop << 16);
            if (complete) {
                p.recs[pos] = make_uint4(ra1, ra2, rfl, 0u);
                fl &= ~LF_RUN; surv = false;
            } else if (kprop == 0u) {
                /* first survivor of an exact observation: go on to the proposal search */
                fast_begin(f, f.a + 1u, n); surv = false;
            } else {
                /* next proposal: sub-stream a+1 from draw 1 (draw 0 was the accept uniform) */
                const uint32_t a = f.a + 1u;
                const uint32_t res = exact_attempt<NC, IV>(a, true, p.y[pos], o.cens, o.og, p, sm, iter, n, smask, upper_at<IV>(p.u, pos));
                surv = res & 1u; k = (int)((res >> 8) & 0xffu); c_jumps += res >> 16;
                this_off = true;
                if (!surv) c_attempts++;
                fast_begin(f, surv ? a : a + 1u, n);
            }
        }
        if (hand && (fl & LF_RUN)) {
            const uint32_t idx = atomicAdd(&p.state->n_items, 1u);
            if (idx < p.item_cap) {
                const uint32_t misc = sm.mh_misc[tid];
                TailItem it; it.y = p.y[pos]; it.og = o.og; it.pos = pos; it.a = f.a; it.cur_a = sm.mh_cur_a[tid];
                it.flags = pack_flags((fl & LF_HAVE) != 0u, (misc >> 8) & 1u, false, o.cens, (int)(misc & 0xffu), misc >> 16);
                it.owner = p.obs_rank;
                p.items[idx] = it; p.found[idx] = FOUND_NONE;
                if constexpr (IV) p.item_u[idx] = p.u[pos];
                atomicAdd(&p.state->counters[PHT_CNT_DEFERRED], 1ull);
                fl &= ~LF_RUN;
            } else a_lim = 0xFFFFFFFFu;          /* no room: the lane keeps the observation */
        }
        __syncwarp();
    }
}

/* block accumulators and per-thread event counts -> global memory */
template <int NC>
__device__ __forceinline__ void flush_block(const SweepParams &p, MhrsSmem<NC> &sm, int n, bool stats, unsigned c_attempts, unsigned c_jumps) {
    const unsigned FULL = 0xffffffffu; const int tid = threadIdx.x;
    __syncthreads();
    if (stats) {
        unsigned long long *gN = reinterpret_cast<unsigned long long *>(p.stats);
        for (int i = tid; i < n * n; i += MHRS_THREADS) if (sm.Nacc[i]) atomicAdd(&gN[i], (unsigned long long)sm.Nacc[i]);
        for (int i = tid; i < n; i += MHRS_THREADS) {
            if (sm.Bacc[i]) atomicAdd(&gN[n * n + i], (unsigned long long)sm.Bacc[i]);
            if (sm.zlo[i]) atomicAdd(&gN[n * n + n + i], sm.zlo[i]);
            if (sm.zhi[i]) atomicAdd(&gN[n * n + 2 * n + i], (unsigned long long)sm.zhi[i]);
        }
    }
    unsigned long long w_attempts = c_attempts, w_jumps = c_jumps;
    for (int o = 16; o > 0; o >>= 1) { w_attempts += __shfl_down_sync(FULL, w_attempts, o); w_jumps += __shfl_down_sync(FULL, w_jumps, o); }
    if ((tid & 31) == 0) { atomicAdd(&p.state->counters[PHT_CNT_ATTEMPTS], w_attempts); atomicAdd(&p.state->counters[PHT_CNT_JUMPS], w_jumps); }
    if (tid == 0 && sm.paths_done) atomicAdd(&p.state->counters[PHT_CNT_PATHS], (unsigned long long)sm.paths_done);
}

/* states that can exit: bit j of smask (the accept tests of eq_Bladt_MHRS.c:66,74 need s[j] != 0) */
template <int NC>
__device__ __forceinline__ void model_scalars(const MhrsSmem<NC> &sm, int n, uint32_t &smask) {
    smask = 0u;
    for (int i = 0; i < n; i++) smask |= (sm.s[i] != 0.0) ? (1u << i) : 0u;
}

/* Kernel 1 of the MHRS sweep: the lane phase (an ordinary launch; its own register budget).
 * IV = true: the instance for sweeps with interval bounds set (SweepParams::u); kernels 1 and 2 have one each, the replay
 * none (it replays an accepted attempt, whose path statistics are those of a right-censored observation). */
template <int NC, bool IV>
__global__ void __launch_bounds__(MHRS_THREADS, MHRS_MIN_BLOCKS) k_mhrs_lanes(const __grid_constant__ SweepParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    MhrsSmem<NC> &sm = *reinterpret_cast<MhrsSmem<NC> *>(smem_raw);
    const int n = p.n;
    const uint32_t iter = p.state->iter;
    const unsigned long long t0 = (blockIdx.x == 0 && threadIdx.x == 0) ? gtimer() : 0ull;
    build_tables(p, sm, n, ModelLayout::make(n, p.m));
    uint32_t smask;
    model_scalars(sm, n, smask);
    const bool per_obs = p.outB != nullptr;
    const uint32_t obs_begin = per_obs ? (uint32_t)p.first : 0u;
    const uint32_t obs_end = per_obs ? (uint32_t)(p.first + p.count) : (uint32_t)p.l_local;
    const uint32_t cap = p.mhrs_cap > 0 ? (uint32_t)p.mhrs_cap : 256u;
    unsigned c_attempts = 0, c_jumps = 0;      /* per thread and sweep: far below 2^32 */
    lane_phase<NC, IV>(p, sm, iter, n, smask, obs_begin, obs_end, cap, c_jumps, c_attempts);
    flush_block(p, sm, n, false, c_attempts, c_jumps);
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&p.state->counters[PHT_CNT_NS_LANE], gtimer() - t0);
}

/* Kernel 2: the tail (cooperative launch: grid barriers between rounds; peer barriers in global rounds). */
template <int NC, bool IV>
__global__ void __launch_bounds__(MHRS_THREADS, MHRS_TAIL_MIN_BLOCKS) k_mhrs_tail(const __grid_constant__ SweepParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cg::grid_group grid = cg::this_grid();
    MhrsSmem<NC> &sm = *reinterpret_cast<MhrsSmem<NC> *>(smem_raw);
    const int n = p.n, tid = threadIdx.x;
    const uint32_t iter = p.state->iter;
    const bool per_obs = p.outB != nullptr;
    const bool multi = p.xw != nullptr && p.obs_world > 1u && !per_obs;
    const uint32_t n_items = p.state->n_items < p.item_cap ? p.state->n_items : p.item_cap;
    if (n_items == 0u && !multi) return;                  /* every observation finished in its lane */
    const bool timekeeper = (blockIdx.x == 0 && tid == 0);
    unsigned long long t_mark = timekeeper ? gtimer() : 0ull;
    build_tables(p, sm, n, ModelLayout::make(n, p.m));
    uint32_t smask;
    model_scalars(sm, n, smask);
    const double *s_model = p.model + ModelLayout::make(n, p.m).s;
    unsigned c_attempts = 0, c_jumps = 0;
    const uint32_t gtid = blockIdx.x * MHRS_THREADS + tid, gsize = gridDim.x * MHRS_THREADS, nwarps = gsize / 32u;

    for (uint32_t i = gtid; i < n_items; i += gsize) p.pend0[i] = i;
    if (gtid == 0) {
        p.state->n_pend[0] = n_items; p.state->n_pend[1] = 0u; p.state->unit_counter = 0ull;
        p.state->any_fail[0] = 0u; p.state->any_fail[1] = 0u;
    }
    grid.sync();
    /* One loop for both kinds of round.  LOCAL: this rank's pending observations, lists double-buffered and
     * compacted every round.  GLOBAL (several GPUs, from K = k_switch on): the observations still pending on any
     * rank, gathered once into every rank's exchange window in a canonical order that never changes (finished
     * items are flagged and skipped), searched by all ranks, advanced by every rank redundantly. */
    /* round 0 offers every pending observation as many attempts as its lane has already spent on it */
    uint32_t K = TAIL_K0; while (K < (uint32_t)p.mhrs_cap && K < TAIL_KMAX) K *= 2u;
    uint32_t rounds = 0u, g0 = 0u, Pg = 0u; int cur = 0, gl_cur = 0; bool global = false;
    const uint32_t W = p.obs_world, me = p.obs_rank, sp = iter & 1u;
    unsigned long long epoch = multi ? p.state->xepoch : 0ull;
    for (;;) {
        const uint32_t *pend = cur ? p.pend1 : p.pend0;
        uint32_t *pend_next = cur ? p.pend0 : p.pend1;
        if (!global) {
            const uint32_t P = p.state->n_pend[cur];
            const bool leave = P == 0u || (multi && K >= p.k_switch && P <= PHT_GCAP);
            if (leave && !multi) break;
            if (leave) {
                /* ---- gather: my pending items into every rank's window (mine included), then the canonical list */
                if (timekeeper) { const unsigned long long t = gtimer(); atomicAdd(&p.state->counters[PHT_CNT_NS_TAIL], t - t_mark); t_mark = t; }
                for (uint32_t r = 0; r < W; r++) {
                    XchgWindow *dst = p.xpeer[r];
                    for (uint32_t i = gtid; i < P; i += gsize) {
                        dst->gitems[sp][me * PHT_GCAP + i] = p.items[pend[i]];
                        if constexpr (IV) dst->gitem_u[sp][me * PHT_GCAP + i] = p.item_u[pend[i]];
                    }
                    if (gtid == 0) dst->gcount[sp][me] = P;
                }
                peer_barrier(grid, p, ++epoch);
                for (uint32_t r = 0; r < W; r++) {
                    const uint32_t c = p.xw->gcount[sp][r] <= PHT_GCAP ? p.xw->gcount[sp][r] : PHT_GCAP;
                    for (uint32_t i = gtid; i < c; i += gsize) p.glist[Pg + i] = r * PHT_GCAP + i;
                    Pg += c;
                }
                if (gtid == 0) {
                    p.state->n_gpend = Pg; p.state->unit_counter = 0ull; p.state->any_fail[0] = 0u; p.state->any_fail[1] = 0u;
                    atomicAdd(&p.state->counters[PHT_CNT_GLOBAL_ITEMS], (unsigned long long)Pg);
                }
                grid.sync();
                global = true; g0 = rounds;
                K = p.k_switch > TAIL_K0 ? p.k_switch : TAIL_K0;
                continue;
            }
        } else if (Pg == 0u || p.state->xdead != 0u) break;
        const uint32_t par = (rounds - g0) & 1u;
        TailView tv;
        if (!global) { tv.items = p.items; tv.pend = pend; tv.found = p.found; tv.P = p.state->n_pend[cur]; tv.u = p.item_u; }
        else { tv.items = p.xw->gitems[sp]; tv.pend = gl_cur ? p.glist + PHT_MAX_WORLD * PHT_GCAP : p.glist; tv.found = p.xw->gfound[par]; tv.P = Pg; tv.u = p.xw->gitem_u[sp]; }
        tv.K = K; tv.global = global; tv.parity = par;
        const unsigned long long tr0 = timekeeper ? gtimer() : 0ull;
        const unsigned att0 = c_attempts, jmp0 = c_jumps;
        tail_search<NC, IV>(tv, p, sm, iter, n, smask, nwarps, c_jumps, c_attempts);
        const unsigned long long tr1 = timekeeper ? gtimer() : 0ull;
        if (rounds < PHT_ROUND_TRACE) {          /* attempts this round ran, over the whole grid (measurement aid) */
            unsigned d = c_attempts - att0;
            for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
            if ((tid & 31) == 0 && d) atomicAdd(&p.state->round_trace[rounds][5], (unsigned long long)d);
            unsigned dj = c_jumps - jmp0;
            for (int o = 16; o > 0; o >>= 1) dj += __shfl_xor_sync(0xffffffffu, dj, o);
            if ((tid & 31) == 0 && dj) atomicAdd(&p.state->round_trace[rounds][7], (unsigned long long)dj);
        }
        if (global) peer_barrier(grid, p, ++epoch); else grid.sync();
        const unsigned long long tr2 = timekeeper ? gtimer() : 0ull;
        /* ---- advance each pending observation's MH state machine (eq_Bladt_MHRS.c:65-101); in a global round every
         * rank advances every item: same inputs, same outcome */
        for (uint32_t i = gtid; i < tv.P; i += gsize) {
            const uint32_t item = tv.pend[i];
            TailItem it = tv.items[item];
            if (it.flags & TI_FIN) continue;
            bool failed;
            if (rounds < PHT_ROUND_TRACE && (!global || it.owner == me)) {      /* attempts the sequential sampler runs of this round's offer */
                const unsigned long long fw = tv.found[item];
                atomicAdd(&p.state->round_trace[rounds][6], fw == FOUND_NONE ? (unsigned long long)K : (unsigned long long)((uint32_t)(fw >> 8) - it.a + 1u));
            }
            const int st = tail_advance(it, tv.found[item], K, p, s_model, iter, failed);
            tv.found[item] = FOUND_NONE;
            if (st != 0 && global) it.flags |= TI_FIN;
            tv.items[item] = it;
            const bool mine = !global || it.owner == me;
            if (st == 2 && mine) { atomicAdd(&p.state->counters[PHT_CNT_ERRORS], 1ull); atomicOr(&p.state->error, 8); }
            if (failed && st == 0) atomicOr(&p.state->any_fail[par], 1u);
            /* a finished observation leaves its record for the replay kernel (the owner's list, the owner's position) */
            if (st != 0 && mine) p.recs[it.pos] = (st == 1) ? make_uint4(it.cur_a, 0u, (it.flags & TI_CUROFF) ? RF_OFF : 0u, 0u) : make_uint4(0u, 0u, RF_SKIP, 0u);
            if (st == 0 && !global) pend_next[atomicAdd(&p.state->n_pend[cur ^ 1], 1u)] = item;
        }
        if (gtid == 0) { if (!global) p.state->n_pend[cur] = 0u; p.state->unit_counter = 0ull; p.state->any_fail[par ^ 1u] = 0u; }
        grid.sync();
        if (global) {
            /* the canonical list without the finished items, in the same order on every rank (one block, ballot scan) */
            uint32_t *next_list = (gl_cur ? p.glist : p.glist + PHT_MAX_WORLD * PHT_GCAP);
            if (blockIdx.x == 0) {
                const int lane = tid & 31, warp = tid >> 5;
                uint32_t outn = 0u;
                for (uint32_t tile = 0; tile < Pg; tile += MHRS_THREADS) {
                    const uint32_t i = tile + tid;
                    uint32_t item = 0u; bool keep = false;
                    if (i < Pg) { item = tv.pend[i]; keep = !(tv.items[item].flags & TI_FIN); }
                    const unsigned bal = __ballot_sync(0xffffffffu, keep);
                    if (lane == 0) sm.scan[warp] = __popc(bal);
                    __syncthreads();
                    uint32_t off = 0u, tot = 0u;
                    for (int w2 = 0; w2 < MHRS_WARPS; w2++) { const uint32_t c = sm.scan[w2]; off += (w2 < warp) ? c : 0u; tot += c; }
                    if (keep) next_list[outn + off + __popc(bal & ((1u << lane) - 1u))] = item;
                    outn += tot;
                    __syncthreads();
                }
                if (tid == 0) p.state->n_gpend = outn;
            }
            grid.sync();
            Pg = p.state->n_gpend; gl_cur ^= 1;
        }
        /* the attempts per observation grow only when some observation needed more than this round offered: with
         * mhit > 1 every pending observation comes back round after round for its next proposal, and a K that kept
         * doubling would bury the round in pools to skip */
        const bool grow = p.state->any_fail[par] != 0u;
        if (timekeeper && rounds < PHT_ROUND_TRACE) {
            unsigned long long *tr = p.state->round_trace[rounds];
            tr[0] += tr1 - tr0; tr[1] += tr2 - tr1; tr[2] += gtimer() - tr2; tr[3] += tv.P; tr[4] += K;
        }
        if (!global) cur ^= 1;
        rounds++;
        if (grow && K < TAIL_KMAX) K *= ((global ? Pg : p.state->n_pend[cur]) <= TAIL_LATE_P) ? TAIL_LATE_GROWTH : TAIL_GROWTH;
        if (K > TAIL_KMAX) K = TAIL_KMAX;
    }
    if (multi && gtid == 0) { p.state->xepoch = epoch; p.state->n_pend[cur] = 0u; }
    if (timekeeper) {
        const unsigned long long t = gtimer();
        atomicAdd(&p.state->counters[global ? PHT_CNT_NS_GLOBAL : PHT_CNT_NS_TAIL], t - t_mark); t_mark = t;
    }
    if (gtid == 0) {
        atomicAdd(&p.state->counters[PHT_CNT_TAIL_ROUNDS], (unsigned long long)rounds);
        if (global) atomicAdd(&p.state->counters[PHT_CNT_GLOBAL_ROUNDS], (unsigned long long)(rounds - g0));
    }
    flush_block(p, sm, n, false, c_attempts, c_jumps);
}

/* Kernel 3: the exact replay of every observation's accepted attempt, with recording on (see replay_phase). */
template <int NC>
__global__ void __launch_bounds__(MHRS_THREADS, MHRS_REPLAY_MIN_BLOCKS) k_mhrs_replay(const __grid_constant__ SweepParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    MhrsSmem<NC> &sm = *reinterpret_cast<MhrsSmem<NC> *>(smem_raw);
    const int n = p.n;
    const uint32_t iter = p.state->iter;
    const unsigned long long t0 = (blockIdx.x == 0 && threadIdx.x == 0) ? gtimer() : 0ull;
    build_tables(p, sm, n, ModelLayout::make(n, p.m));
    const bool per_obs = p.outB != nullptr;
    const uint32_t obs_begin = per_obs ? (uint32_t)p.first : 0u;
    const uint32_t obs_end = per_obs ? (uint32_t)(p.first + p.count) : (uint32_t)p.l_local;
    unsigned c_jumps = 0;
    replay_phase(p, sm, iter, n, obs_begin, obs_end, c_jumps);
    flush_block(p, sm, n, !per_obs, 0u, c_jumps);
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&p.state->counters[PHT_CNT_NS_REPLAY], gtimer() - t0);
}

/* ------------------------------------------------------------------------------------------ host side */
template <int NC, bool IV>
static int grid_blocks_of(int device, int *lane_blocks, int *tail_blocks, int *replay_blocks) {
    int a = 0, b = 0, c = 0, sms = 0;
    const size_t smem = sizeof(MhrsSmem<NC>);
    if (cudaFuncSetAttribute(k_mhrs_lanes<NC, IV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(k_mhrs_tail<NC, IV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, k_mhrs_lanes<NC, IV>, MHRS_THREADS, smem) != cudaSuccess) return -1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, k_mhrs_tail<NC, IV>, MHRS_THREADS, smem) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(k_mhrs_replay<NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c, k_mhrs_replay<NC>, MHRS_THREADS, smem) != cudaSuccess) return -1;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return -1;
    *lane_blocks = a * sms; *tail_blocks = b * sms; *replay_blocks = c * sms;
    return (a > 0 && b > 0 && c > 0) ? 0 : -1;
}
/* grid sizes: every SM full of resident blocks of each kernel (persistent warps; the tail launch is cooperative).  The IV
 * instances get grids of their own: their register counts need not be those of the plain ones. */
int pht_mhrs_grid_blocks(int device, int n, bool iv, int *lane_blocks, int *tail_blocks, int *replay_blocks) {
    if (iv) {
        if (n <= 8) return grid_blocks_of<8, true>(device, lane_blocks, tail_blocks, replay_blocks);
        if (n <= 16) return grid_blocks_of<16, true>(device, lane_blocks, tail_blocks, replay_blocks);
        return grid_blocks_of<32, true>(device, lane_blocks, tail_blocks, replay_blocks);
    }
    if (n <= 8) return grid_blocks_of<8, false>(device, lane_blocks, tail_blocks, replay_blocks);
    if (n <= 16) return grid_blocks_of<16, false>(device, lane_blocks, tail_blocks, replay_blocks);
    return grid_blocks_of<32, false>(device, lane_blocks, tail_blocks, replay_blocks);
}
size_t pht_mhrs_smem_bytes(int n) {
    return n <= 8 ? sizeof(MhrsSmem<8>) : (n <= 16 ? sizeof(MhrsSmem<16>) : sizeof(MhrsSmem<32>));
}

template <int NC, bool IV>
static cudaError_t launch_of(const SweepParams &p, int lane_blocks, int tail_blocks, int replay_blocks, cudaStream_t st) {
    SweepParams q = p;
    void *args[] = { &q };
    const size_t smem = sizeof(MhrsSmem<NC>);
    k_mhrs_lanes<NC, IV><<<lane_blocks, MHRS_THREADS, smem, st>>>(q);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    e = cudaLaunchCooperativeKernel((const void *)k_mhrs_tail<NC, IV>, dim3(tail_blocks), dim3(MHRS_THREADS), args, smem, st);
    if (e != cudaSuccess) return e;
    k_mhrs_replay<NC><<<replay_blocks, MHRS_THREADS, smem, st>>>(q);
    return cudaGetLastError();
}
/* the IV instance runs when the sweep has interval bounds (p.u != nullptr), the plain one otherwise */
cudaError_t pht_launch_mhrs(const SweepParams &p, int lane_blocks, int tail_blocks, int replay_blocks, cudaStream_t st) {
    if (p.u != nullptr) {
        if (p.n <= 8) return launch_of<8, true>(p, lane_blocks, tail_blocks, replay_blocks, st);
        if (p.n <= 16) return launch_of<16, true>(p, lane_blocks, tail_blocks, replay_blocks, st);
        return launch_of<32, true>(p, lane_blocks, tail_blocks, replay_blocks, st);
    }
    if (p.n <= 8) return launch_of<8, false>(p, lane_blocks, tail_blocks, replay_blocks, st);
    if (p.n <= 16) return launch_of<16, false>(p, lane_blocks, tail_blocks, replay_blocks, st);
    return launch_of<32, false>(p, lane_blocks, tail_blocks, replay_blocks, st);
}
