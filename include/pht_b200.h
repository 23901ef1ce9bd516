/*
 * pht_b200.h -- C ABI of libpht_b200.so, the B200-native Gibbs engine that sits
 * behind PhaseType's native entry point.  Plain pointers and sizes only.
 *
 * Layer 1 is the drop-in: the exact routine the R package registers
 * (reference src/PHT_MCMC_Aslett.h:1-3, registered as a 15-argument .C routine
 * in src/Registrations.c:6-14 and called from R/phtMCMC.R:83, R/phtMCMC2.R:73).
 * Layer 2 is the engine API LJMA_Gibbs itself is written on; tests and
 * bench.py use it to keep data resident, shard observations over GPUs and read
 * per-observation statistics for parity checks.
 *
 * There is no CPU fallback: every entry point fails (non-zero return and a
 * message from pht_last_error()) when no CUDA device is usable.
 */
#ifndef PHT_B200_H
#define PHT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ layer 1 */

/* Replaces reference src/PHT_MCMC_Aslett.c:104 (same name, same 15 arguments,
 * same meaning: documented at src/PHT_MCMC_Aslett.c:72-103).  R's `censored` has
 * no slot for an upper bound, so interval-censored data go through layer 2
 * (pht_engine_set_upper), not through this routine.  `res` (it x m,
 * column-major) is fully overwritten; row 0 is the start value.  Diagnostics go
 * through Rprintf; nothing is signalled (void), as in the reference.
 * Engine knobs that have no slot in the 15 arguments come from the environment:
 *   PHT_B200_SEED     (decimal/hex uint64; default: drawn from unif_rand())
 *   PHT_B200_DEVICE   (CUDA ordinal, default 0)
 *   PHT_B200_GRAPH    (0: launch the sweep's kernels directly instead of replaying a CUDA graph)
 *   PHT_B200_MHRS_CAP (attempts a lane tries before handing an observation to the cooperative tail; default 32..1024 by shard size)
 *   PHT_B200_GPUS     (devices to fan out over, starting at PHT_B200_DEVICE; default: one per 2^19 observations, at most
 *                      all visible.  One host thread + one engine per device; the all-reduce of the statistics and the
 *                      global MHRS tail run through peer memory inside the sweep's kernels; the chain does not depend
 *                      on the number of devices)
 *   PHT_B200_NCCL     (1: all-reduce the statistics with ncclAllReduce instead of the engine's own peer-memory kernel)
 *   PHT_B200_ZBITS    (fractional bits of the fixed-point sojourn totals; default from sum(y))
 *   PHT_B200_SEED_EXACT (use PHT_B200_SEED as is even with start values given; default: the start vector is mixed into
 *                      the key so that a resumed run does not replay the streams of the run it continues)
 *   PHT_B200_BETA     (comma-separated Dirichlet prior of the start distribution, n values: switches its update on;
 *                      PHT_B200_PI0 = comma-separated initial pi, default e1; PHT_B200_PI_OUT = file that receives the
 *                      it x n draws as text, one row per iteration -- `res` has no columns for them)
 *   PHT_B200_NO_POOL  (1: plain cudaMalloc/cudaFree for the large per-call buffers instead of the devices' memory pools,
 *                      which keep the memory cached between calls -- see pht_release_device_memory)
 *   PHT_B200_TIMING   (1: stage times of the call's set-up on stderr) */
void LJMA_Gibbs(int *it, int *mhit, int *method, int *n, int *m, double *nu, double *zeta,
                int *T, double *C, double *y, int *l, int *censored, double *start,
                int *silent, double *res);

/* ------------------------------------------------------------------ layer 2 */

#define PHT_METHOD_MHRS 1   /* reference src/PHT_MCMC_Aslett.c:69-71 */
#define PHT_METHOD_ECS  2
#define PHT_METHOD_DCS  4
/* The two sampler variants the reference compiles but never dispatches (SURVEY.md section 8(f)1), reachable here behind
 * two further bits of the same mask; they have the lowest priority, so every mask the reference understands keeps its
 * meaning.  Both take `mhit` like MHRS. */
#define PHT_METHOD_MHS_HOBOLTH 8    /* LJMA_MHsample_Hobolth, src/Simulate_AbsCTMC_gt_Hobolth_DCS.c:268-355: Hobolth paths
                                       conditioned on the exit set {j : s_j > 0} + independence MH; censoring ignored by
                                       the chain sampler (the MH step is skipped for a censored observation) */
#define PHT_METHOD_MHS_ASLETT 16    /* LJMA_MHsample_Aslett (reverse = 0), src/Simulate_AbsCTMC_eq_Aslett_DCS.c:49-143: the
                                       Aslett-DCS "alive at y" sampler for every observation + independence MH */
/* The uniformisation path sampler (Hobolth & Stone 2009, section 3.3; the engine's own, no reference counterpart): every
 * path is drawn from its exact conditional law given the data, for any sub-generator (a Jordan block or a complex
 * spectrum included), through the uniformised chain R = I + S/lambda, lambda = max_i -S_ii, and a table of its powers
 * built once per sweep.  Exact, right-censored, interval-censored (pht_engine_set_upper) and left-censored (y = 0 with a
 * finite bound) observations; the start state is drawn from its conditional law too, so the start-distribution update
 * (pht_engine_set_pi with beta) works with it.  Lowest priority of the mask; `mhit` is not used.  The table holds
 * PHT_UNIF_CAP = 4096 powers (33 MB at n = 32): an observation whose lambda y (or lambda (u - y)) needs more raises error
 * bit 256.  Delayed entry (left-truncated observations, pht_engine_set_entry) is this method's alone.  (Bit 32 stays
 * unassigned.) */
#define PHT_METHOD_UNIF 64
#define PHT_MAX_PHASES  32

typedef struct pht_engine pht_engine;

typedef struct pht_config {
    int n;                /* transient phases, 1..PHT_MAX_PHASES */
    int m;                /* number of rate parameters */
    int method;           /* bit mask as in the reference; priority MHRS > DCS > ECS (> 8 > 16 > 64, the engine's own) */
    int mhit;             /* Metropolis-Hastings proposals per exact observation (MHRS) */
    const int *T;         /* (n+1)^2 column-major: 0 = structural zero, v>=1 = parameter index */
    const double *C;      /* (n+1)^2 constant multipliers */
    const double *nu;     /* m Gamma shapes */
    const double *zeta;   /* m Gamma rates */
    uint64_t seed;        /* Philox key of the chain */
    int device;           /* CUDA ordinal */
    int rank, world;      /* this engine holds observations rank, rank+world, ... of the global set */
    int zbits;            /* fractional bits of the fixed-point sojourn totals (pht_choose_zbits) */
    int mhrs_cap;         /* attempts a lane tries before handing an observation to the cooperative tail; 0 = default
                             (8 x observations per resident lane, as a power of two between 32 and 1024) */
    int use_graph;        /* capture the sweep in a CUDA graph (1) or launch kernels directly (0) */
} pht_config;

const char *pht_last_error(void);
int pht_device_count(void);
/* The large per-call device buffers come from the devices' stream-ordered memory pools and stay cached there after
 * a call (the next call reuses them; PHT_B200_NO_POOL=1 switches this off).  This hands the cached memory back. */
int pht_release_device_memory(void);

/* 62 - ceil(log2(16 * sum_y)): every per-state total fits an int64 with headroom */
int pht_choose_zbits(double sum_y_global);

/* y_local / cens_local: host arrays of the l_local observations this rank owns
 * (global index of local k is rank + k*world); copied to the device. */
int pht_engine_create(pht_engine **out, const pht_config *cfg, const double *y_local,
                      const int *cens_local, long l_local);
void pht_engine_destroy(pht_engine *e);

/* multi-GPU, one process per GPU, statistics all-reduced by NCCL: rank 0 calls pht_comm_unique_id, the 128 bytes
 * travel over the launcher's own channel, every rank calls pht_engine_comm_init.  Not needed when the engines'
 * exchange windows are attached (below): the all-reduce then runs through them (k_allreduce_peer), unless
 * PHT_B200_NCCL=1 asks for NCCL. */
int pht_comm_unique_id(void *id128);
int pht_engine_comm_init(pht_engine *e, const void *id128);

/* Several GPUs of one box: each engine owns an exchange window in device memory that its peers write into over NVLink.
 * Two things run through it, inside the sweep's own kernels (no host, no library call): the per-sweep all-reduce of
 * the statistics block (every method), and for MHRS the deepest part of the rejection tail (observations that need
 * 10^5..10^8 attempts), which all ranks search together.
 * pht_engine_peer_handle writes an opaque PHT_PEER_HANDLE_BYTES handle for it, the launcher gathers the handles of
 * all ranks (rank order) and every rank calls pht_engine_peer_attach with the concatenation.  Works between
 * processes (CUDA IPC) and between engines of one process (direct peer access).  A multi-rank run needs either the
 * windows or an NCCL communicator (pht_engine_comm_init) for its statistics; with NCCL only, the MHRS tail rounds stay
 * local to each rank and the chain is the same, only slower to finish. */
#define PHT_PEER_HANDLE_BYTES 128
int pht_engine_peer_handle(pht_engine *e, void *handle);
int pht_engine_peer_attach(pht_engine *e, const void *handles);

/* parameter vector (length m) the next sweep starts from, and the index that sweep gets */
int pht_engine_set_theta(pht_engine *e, const double *theta, uint32_t next_iter);
int pht_engine_get_theta(pht_engine *e, double *theta);

/* Start distribution.  The reference fixes pi = e1 and leaves its update as FIX ME (src/PHT_MCMC_Aslett.c:190-193) although
 * R passes a Dirichlet prior `beta` down to the wrapper (R/phtMCMC2.R:20-21).  pi (n values, may be NULL: keep) sets the
 * distribution the samplers start their paths from; beta (n positive values, may be NULL: no update) switches on the
 * conjugate update pi | paths ~ Dirichlet(beta + B) at the end of every sweep (methods MHRS and 64 only: a rejection
 * sampler started from pi, and the uniformisation sampler, draw the start state from its conditional law given y; the
 * reference's ECS and DCS samplers draw it from pi itself, which is exact for the degenerate pi the reference uses and
 * nothing else).  pht_engine_pi_rows returns
 * the draws of the last pht_engine_run (rows x n, row-major). */
int pht_engine_set_pi(pht_engine *e, const double *pi, const double *beta);
int pht_engine_get_pi(pht_engine *e, double *pi);
int pht_engine_pi_rows(pht_engine *e, int rows, double *out);

/* Interval-censored observations (methods MHRS and 64): the absorption time of local observation k is known to lie in
 * [y_k, u_k].  upper_local holds one u per local observation, in the order of y_local; +INFINITY means no bound
 * (exact or right-censored as before, with the same results bit for bit).  A finite u needs the censoring flag and
 * u > y.  Paths are drawn from their law given y <= T <= u by the same rejection sampler (an attempt survives when it
 * is absorbed in [y, u]); their statistics are those of a right-censored path.  Interval paths end by u, so the
 * configured zbits may be at most pht_choose_zbits(sum over the observations of max(y, u)).  NULL clears the bounds.
 * Every rank of a multi-rank run sets bounds (or none) before the exchange windows are attached.  Refused for ECS,
 * DCS and the two MH variants.  Method 64 draws the path given y < T <= u directly (no rejection: the cost does not
 * depend on the width of the interval) and also takes y = 0 with a finite u: a failure before the first inspection
 * (left-censored); MHRS needs y > 0. */
int pht_engine_set_upper(pht_engine *e, const double *upper_local);

/* Delayed entry, also called left truncation (method 64 only): local observation k entered the study at age a_k because it
 * was still working then (a component bought used, a patient enrolled at some age), so the sample holds only units with
 * T > a_k and each contributes L_k / S(a_k).  entry_local holds one a per local observation, in the order of y_local; 0
 * means no truncation (the results are those without entry ages, bit for bit); NULL clears the ages.  Every sweep draws,
 * per observation with a > 0, the number M of units of its kind lost before a (M | theta ~ Geometric, P(M = k) =
 * F(a)^k S(a)) and each lost unit's path given absorption in (0, a]; their start states, transitions and sojourns join
 * the sweep statistics, which keeps the update conjugate (Dempster, Laird & Rubin 1977).  The observations' own paths
 * are drawn as before.  Refused: NaN, +-inf, a < 0, a > y (a left-censored record, y = 0, takes no entry age), a call
 * after the exchange windows are attached (every rank sets ages, or none, before), and a zbits above
 * pht_choose_zbits(sum over the observations of max(y, u) + a).  That sum counts one ghost path per truncated observation;
 * the fixed point holds at least 32 times it per sweep, so ghost time up to ~30 times one ghost per observation still
 * fits, and beyond that error word 2 reports the overflow.  Error bit 1024:
 * S(a) underflowed, or a ghost count above 2^20 (the model leaves almost no survival at that age).  It ends the run, and
 * it is a draw: an observation whose S(a) at the chain's current theta is ~1e-6 raises it with probability
 * exp(-2^20 S(a)) ~ 0.35 per sweep, so entry ages far in the model's tail (a unit entering long after nearly all of its
 * kind have failed) can stop a chain mid-run even when early sweeps pass.  Refused for MHRS,
 * ECS, DCS and the two MH variants. */
int pht_engine_set_entry(pht_engine *e, const double *entry_local);

/* Several chains in one engine (method 64 only).  Chain c is, bit for bit, the chain a single-chain engine created with
 * Philox key keys[c] draws from the same theta, pi, prior, data, bounds and next_iter: every sweep statistic is an integer
 * sum, and every chain runs the same table, path and update code on its own model block with its own key.  The chains
 * share the observations, the bounds and the sorted layout; each has its own model block, statistics block, 33 MB table
 * (at n = 32) and result rows.  One sweep builds the chains' tables side by side (one block each) and the path kernel
 * spreads every chain's observations over the GPU, so at small shards C chains cost about what one does.
 * pht_engine_set_chains: keys holds `chains` Philox keys, NULL = the configured seed + c.  Every chain starts from the
 * engine's current theta and pi; chains = 1 returns to the single-chain engine, whose results are those of an engine that
 * never called it.  With several chains the existing calls keep their meaning for chain 0 (pht_engine_get_theta, run's
 * out, pht_engine_pi_rows, pht_engine_get_model; the parity hooks pht_engine_sweep_stats and pht_engine_paths run chain
 * 0 alone), while pht_engine_set_theta and pht_engine_set_pi set every chain.  Refused: any method but 64, world > 1 (the
 * all-reduce carries one chain's statistics), entry ages (pht_engine_set_entry, in either order), chains outside
 * 1..PHT_MAX_CHAINS, duplicate keys, and a failed allocation (the engine then stays as it was).
 * pht_engine_set_chain_theta / pht_engine_get_chain_theta: one theta per chain (chains x m, row-major); set also gives
 * the next sweep index next_iter, as pht_engine_set_theta does.
 * pht_engine_chain_rows: the draws of the last pht_engine_run, theta as chains x rows x m and pi as chains x rows x n
 * (either may be NULL; pi needs the prior set, pht_engine_set_pi with beta). */
#define PHT_MAX_CHAINS 1024
int pht_engine_set_chains(pht_engine *e, int chains, const uint64_t *keys);
int pht_engine_set_chain_theta(pht_engine *e, const double *theta, uint32_t next_iter);
int pht_engine_get_chain_theta(pht_engine *e, double *theta);
int pht_engine_chain_rows(pht_engine *e, int rows, double *theta_out, double *pi_out);

/* Groups of observations with their own generator structure, sharing one parameter vector (method 64 only): treatment and
 * control arms, two hospitals, two production lots.  Group g's structure (T_g, C_g) maps the engine's m parameters theta
 * (with the engine's nu and zeta; m <= n(n+1) as pht_engine_create takes it) onto its own n-phase generator, e.g. a
 * Coxian whose progression rates are shared and whose exit rates are per group.  The model stays conjugate: parameter k's full conditional is a Gamma whose statistics
 * sum, over the groups in ascending order, every cell of the group's structure that carries k (within a group in the order
 * a single structure uses, the reference's z / C gather included).  pi is one vector per chain, shared by all groups; its
 * Dirichlet update sums the start-state counts of every group.  Each observation's path is drawn on its own group's model
 * and is, bit for bit, the path an engine configured with (T_g, C_g) draws for it from the same key, sweep, theta and pi.
 * pht_engine_set_groups: T and C hold G structures of (n+1)^2 entries each, column-major like pht_config::T / C; group_local
 * holds the group 0..G-1 of every local observation, in the order of y_local.  T = NULL returns to the configured structure
 * (G, C and group_local are then ignored).  G = 1 with the configured T and C and every observation in group 0 is the
 * engine as it was, bit for bit.  Every chain keeps its theta and pi.  The sweep builds one table per group, spanning that
 * group's own observations, and one per chain; chains x G tables in all (33 MB each at n = 32).
 * pht_engine_group_stats: as pht_engine_sweep_stats (chain 0, one sweep, no update), per group: N (G x n*n), B (G x n),
 * zfix (G x n); pht_engine_sweep_stats returns their sum over the groups.  pht_engine_paths records each observation's
 * path drawn on its own group's model, in upload order.
 * Refused, each with its own message and leaving the engine as it was: any method but 64; world > 1 (the all-reduce carries
 * one statistics block); G > 1 with entry ages set (pht_engine_set_entry, in either order: the ghost paths are drawn on
 * one model); G outside 1..PHT_MAX_GROUPS or chains x G above PHT_MAX_CHAINS (pht_engine_set_chains checks the same
 * product); a T_g that pht_engine_create would refuse; a parameter used by no group's structure; a group id out of range;
 * a failed allocation. */
#define PHT_MAX_GROUPS 64
int pht_engine_set_groups(pht_engine *e, int G, const int *T, const double *C, const int *group_local);
int pht_engine_group_stats(pht_engine *e, long long *N, long long *B, long long *zfix);

/* run `nsweeps` Gibbs sweeps; row r of out (nsweeps x m, row-major) is the draw of sweep r.
 * out may be NULL (results stay on the device; fetch later with pht_engine_get_theta). */
int pht_engine_run(pht_engine *e, int nsweeps, double *out);
/* asynchronous halves of pht_engine_run for timing with CUDA events */
int pht_engine_enqueue(pht_engine *e, int nsweeps);
int pht_engine_sync(pht_engine *e);
/* measurement aid: write `bytes` of scratch (larger than L2) on the sweep stream before every sweep, so that no sweep
 * finds its observations in L2 from the previous one; 0 switches it off (default) */
int pht_engine_set_l2_flush(pht_engine *e, unsigned long long bytes);
/* device time in ms of the sweeps enqueued by the last pht_engine_enqueue (after sync): all of them, and the path kernels
 * per sweep (with the ghost pass of delayed entry, pht_engine_set_entry; measured only without the CUDA graph) */
int pht_engine_last_ms(pht_engine *e, float *total_ms, float *path_kernel_ms);

/* parity hooks ------------------------------------------------------------- */
/* sufficient statistics of ONE sweep at the current parameters without updating them:
 * N (n*n), B (n) counts and z (n) totals of this rank's shard (before any all-reduce) */
int pht_engine_sweep_stats(pht_engine *e, long long *N, long long *B, long long *zfix);
/* per-observation statistics for local observations [first, first+count): B[count],
 * N[count*n*n] (int32), z[count*n]; same kernels, recording to memory instead of reducing */
int pht_engine_paths(pht_engine *e, long first, long count, int *B, int *N, double *z);
/* delayed entry (pht_engine_set_entry): the ghost counts M[count] of local observations [first, first+count) in upload
 * order, and when B is not NULL all total = sum M ghost paths in (observation, ghost index) order: B[total],
 * N[total*n*n] (int32), z[total*n]; same kernels as a sweep, recording to memory.  Without entry ages M is all zero. */
int pht_engine_entry_paths(pht_engine *e, long first, long count, int *M, long total, int *B, int *N, double *z);
/* override the spectral data the ECS/DCS kernels use (evals n, Q n*n, Qinv n*n); NULL restores the device solver;
 * refused for method 64, which uses none */
int pht_engine_set_spectral(pht_engine *e, const double *evals, const double *Q, const double *Qinv);
/* current model matrices as the kernels see them (each may be NULL) */
int pht_engine_get_model(pht_engine *e, double *S, double *s, double *P, double *Pfull,
                         double *evals, double *Q, double *Qinv);
/* event counters accumulated since creation (index meaning: PHT_CNT_*) */
enum { PHT_CNT_PATHS = 0, PHT_CNT_ATTEMPTS, PHT_CNT_JUMPS, PHT_CNT_DENS_EVALS, PHT_CNT_ENV_UPDATES,
       PHT_CNT_BRENT_EVALS, PHT_CNT_ARMS_CALLS, PHT_CNT_METROP_REJECTS, PHT_CNT_NONFINITE,
       PHT_CNT_DEFERRED, PHT_CNT_TAIL_ROUNDS, PHT_CNT_ERRORS, PHT_CNT_LAUNCHES,
       PHT_CNT_NS_LANE, PHT_CNT_NS_TAIL, PHT_CNT_NS_REPLAY,   /* device-timer ns spent in the MHRS kernel phases */
       PHT_CNT_NS_GLOBAL,                                      /* ... and in the tail rounds searched by all GPUs together */
       PHT_CNT_NS_XWAIT,                                       /* part of NS_GLOBAL spent in barriers between the GPUs */
       PHT_CNT_GLOBAL_ROUNDS, PHT_CNT_GLOBAL_ITEMS,            /* global tail: rounds run, observations gathered */
       PHT_CNT_COUNT = 20 };
int pht_engine_counters(pht_engine *e, unsigned long long *out);
/* MHRS tail, per round number (accumulated since creation): ns searching, ns at the barrier after the search, ns
 * advancing, sum of pending observations, sum of attempts offered per observation,
 * attempts actually run in the round (all warps), attempts the sequential sampler needs of it, jump-steps run;
 * out: PHT_ROUND_TRACE x 8 words */
#define PHT_ROUND_TRACE 48
int pht_engine_round_trace(pht_engine *e, unsigned long long *out);

/* measurement helpers ------------------------------------------------------- */
/* dependent-chain FP64 FMA microbenchmark: achieved FMA instructions per second (all SMs) */
int pht_fp64_fma_rate(int device, double *fma_per_s);

#ifdef __cplusplus
}
#endif
#endif /* PHT_B200_H */
