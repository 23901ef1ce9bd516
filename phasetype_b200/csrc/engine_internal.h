/*
 * engine_internal.h -- data layout shared by the engine (engine.cu) and its kernels.
 *
 * HBM layout (all per engine = per GPU):
 *   y[l_local]      fp64   observations of this rank's shard (global index rank + k*world)
 *   cens[l_local]   uint8  right-censoring flags (the ABI's int32 is repacked at upload)
 *   unif[]          fp64   method 64 only: the uniformisation table (pht_unif.h; 33 MB at n = 32)
 *   u[l_local]      fp64   MHRS and method 64 only, when interval bounds are set (pht_engine_set_upper): upper bound of each
 *                          censored observation's absorption time, +inf = none; a copy in the decreasing-y layout
 *   entry[]         fp64   method 64 only, when entry ages are set (pht_engine_set_entry): a per observation in upload
 *                          order; the truncated ones (a > 0) as a list by decreasing a with their local indices, ghost
 *                          counts and offsets; the entry tables (2 x PHT_UNIF_CAP)
 *   model[]         fp64   the per-sweep model block, offsets from ModelLayout (< 70 KB at n = 32);
 *                          rebuilt on the device every sweep, copied to shared memory by the path kernels
 *   stats[]         int64  N (n*n) | B (n) | z fixed point in two limbs (2n) | error count: the only data that crosses NVLink
 *   state           DevState: sweep index, work counters, event counters, error word
 * Method 64 with several chains (pht_engine_set_chains) repeats model[], stats[] and unif[] once per chain, chain-major with
 * chain 0 first, and adds the chains' Philox keys and observation counters; observations, bounds and the sorted layout
 * stay shared.
 * Method 64 with groups (pht_engine_set_groups) repeats them once per (chain, group) unit, block c G + g (chain-major, so
 * block c is chain c when G = 1), each unit with its own observation counter; T, C and the parameter -> cell CSR hold one
 * structure per group, and the production layout sorts the observations by group, then by decreasing y.
 *   items/pend/...  MHRS tail work lists (see k_mhrs.cu)
 */
#ifndef PHT_ENGINE_INTERNAL_H
#define PHT_ENGINE_INTERNAL_H

#include <stdint.h>
#include <cuda_runtime.h>
#include "../../include/pht_b200.h"
#include "pht_philox.h"

#define PHT_NMAX PHT_MAX_PHASES

/* offsets in doubles inside the model block */
struct ModelLayout {
    int n, m;
    int S, s, scale, P, Pfull, cum, pi, evals, Q, Qinv, Qinv_s, Qinv_1, TT, theta, evals_im, total;
    __host__ __device__ static ModelLayout make(int n, int m) {
        ModelLayout L; int o = 0;
        L.n = n; L.m = m;
        L.S = o; o += n * n;
        L.s = o; o += n;
        L.scale = o; o += n;                 /* 1.0 / -S[j,j]: the rexp() scale of state j */
        L.P = o; o += n * n;
        L.Pfull = o; o += n * (n + 1);
        L.cum = o; o += (n + 1) * (n + 1);   /* row j<n: running sums of Pfull[j,0..n]; row n: running sums of pi */
        L.pi = o; o += n;
        L.evals = o; o += n;
        L.Q = o; o += n * n;
        L.Qinv = o; o += n * n;
        L.Qinv_s = o; o += n;
        L.Qinv_1 = o; o += n;
        L.TT = o; o += (n + 1) * (n + 1);
        L.theta = o; o += m;
        L.evals_im = o; o += n;              /* +b, -b on the two entries of a complex pair a +- ib, else 0 (pht_eigen.h) */
        L.total = o;
        return L;
    }
};

/* stats block: int64 [ N: n*n | B: n | zlo: n | zhi: n | errors: 1 ].  The fixed-point sojourn total of state i is
 * zhi[i] 2^32 + zlo[i]: every path adds the low 32 bits of its contribution to zlo and the rest to zhi, so the
 * accumulated total cannot wrap (each limb stays far inside 64 bits for 2^32 paths) and k_update can tell exactly
 * whether it still fits the int64 the conjugate update works with.  The last word counts ranks with a raised
 * error word, so that after the all-reduce every rank stops together. */
__host__ __device__ inline int stats_len(int n) { return n * n + 3 * n + 1; }
__device__ __forceinline__ void pht_zfix_add(unsigned long long *zlo, long long *zhi, int i, long long fixed) {
    atomicAdd(&zlo[i], (unsigned long long)fixed & 0xffffffffull);
    atomicAdd(reinterpret_cast<unsigned long long *>(&zhi[i]), (unsigned long long)(fixed >> 32));
}

/* one MHRS observation handed from the lane phase to the cooperative tail.  It carries everything a search of its
 * attempts needs (y, flag, global index), so any GPU of the box can run any of its attempts (global tail rounds). */
struct TailItem {
    double y;
    uint32_t og;          /* global observation index (Philox counter word 2) */
    uint32_t pos;         /* position in the owner's y/cens arrays (for the replay of the accepted attempt) */
    uint32_t a;           /* first attempt index of the current search */
    uint32_t cur_a;       /* attempt index of the accepted draw so far */
    uint32_t flags;       /* bit0 have_cur, bit1 cur_off, bit2 off (for attempt a), bit3 censored, bit4 finished,
                             bits 8..15 cur_pre, bits 16..31 proposals done */
    uint32_t owner;       /* rank that holds the observation */
};
#define TI_HAVE 1u
#define TI_CUROFF 2u
#define TI_OFF 4u
#define TI_CENS 8u
#define TI_FIN 16u

/* Peer-exchange window: one per engine, in device memory, mapped into every other rank of the run (direct peer
 * pointers inside one process, CUDA IPC between processes).  The MHRS kernels of all ranks use it to search the
 * deepest part of the rejection tail together: peers WRITE into it over NVLink (items, surviving attempts, barrier
 * flags), its owner only reads it locally. */
#define PHT_MAX_WORLD 16
#define PHT_GCAP 2048                     /* observations one rank can contribute to a global tail */
#define PHT_STATS_MAX (PHT_NMAX * PHT_NMAX + 3 * PHT_NMAX + 1)
struct XchgWindow {
    /* all-reduce of the statistics block (k_allreduce_peer, every method): rank r stores its block into slot r of
     * every window and raises sflags[r]; double buffered by the parity of the all-reduce count */
    unsigned long long sflags[2][PHT_MAX_WORLD];
    long long sstats[2][PHT_MAX_WORLD][PHT_STATS_MAX];
    /* global MHRS tail */
    unsigned long long flags[PHT_MAX_WORLD];                      /* flags[r]: last barrier epoch rank r arrived at */
    unsigned long long gfound[2][PHT_MAX_WORLD * PHT_GCAP];        /* lowest surviving attempt per item, by round parity */
    uint32_t gcount[2][PHT_MAX_WORLD];                             /* items contributed by rank r, by sweep parity */
    TailItem gitems[2][PHT_MAX_WORLD * PHT_GCAP];                  /* the gathered items, by sweep parity */
    /* upper bounds u of the gathered items (interval-censored observations, k_mhrs.cu IV instance): kept apart so that
     * TailItem stays 32 bytes and no offset above moves; 512 KiB */
    double gitem_u[2][PHT_MAX_WORLD * PHT_GCAP];
};

struct DevState {
    uint32_t iter;             /* index of the sweep about to run (Philox counter word 3) */
    uint32_t first_assembly;   /* 1: diagonals summed in ascending column order (start values) */
    uint32_t res_row;          /* next row of the device result buffer */
    int error;                 /* sticky error word */
    unsigned long long next_obs;      /* lane-phase work counter */
    /* MHRS tail */
    unsigned long long unit_counter;
    uint32_t n_items;          /* items appended by the lane phase */
    uint32_t n_pend[2];        /* pending list sizes (double buffered) */
    uint32_t n_done;           /* (unused) */
    unsigned long long replay_next;   /* MHRS replay kernel: next record to hand out */
    uint32_t any_fail[2];      /* MHRS tail, by round parity: some pending observation found no surviving attempt */
    uint32_t n_gpend;          /* global tail: items not finished yet */
    uint32_t xdead;            /* a peer barrier timed out: no further waiting */
    unsigned long long xepoch; /* barrier epochs completed (monotonic over the life of the engine) */
    unsigned long long sepoch; /* peer all-reduces completed (monotonic over the life of the engine) */
    unsigned long long counters[PHT_CNT_COUNT];
    /* measurement aid: per tail round (index = round number, accumulated over sweeps) the device-timer ns block 0 spent
     * searching / waiting at the barrier after the search / advancing, and the sum of pending items and of K */
    unsigned long long round_trace[PHT_ROUND_TRACE][8];
    uint32_t update_ticket;    /* k_update blocks (one per chain) that have finished; the last one advances the sweep */
};

struct SweepParams {
    /* data */
    const double *y; const uint8_t *cens; long l_local; uint32_t obs_rank, obs_world;
    const uint32_t *perm;      /* position in y/cens -> local observation index; nullptr = identity (y-sorted layout) */
    /* model + state */
    double *model; long long *stats; DevState *state;
    int n, m, mhit, zbits;
    uint32_t k0, k1;           /* Philox key */
    pht_roundkeys rk;          /* its ten round keys (constant-bank operands of the path kernels) */
    /* MHRS tail lists */
    TailItem *items; uint32_t *pend0, *pend1, *done; unsigned long long *found; uint32_t item_cap;
    int mhrs_cap;
    uint4 *recs;               /* MHRS: one 16-byte record per observation position, written by whichever kernel finishes the
                                  observation's search (lanes or tail), read by the replay kernel */
    uint32_t *glist;           /* global tail: the gathered items in canonical (rank-major) order */
    XchgWindow *xw;            /* this rank's exchange window; nullptr = tail rounds stay local */
    XchgWindow *xpeer[PHT_MAX_WORLD];   /* every rank's window as mapped on this device (xpeer[rank] == xw) */
    uint32_t k_switch;         /* attempts per observation and round from which the tail goes global */
    /* per-observation recording (parity mode); all NULL in production */
    int *outB, *outN; double *outz; long first, count;
    /* interval-censored observations (read by the IV instance of the MHRS kernels only; nullptr = no bounds set):
     * u per position, same layout as y, +inf where there is no bound; and the bound of each tail item, indexed like items */
    const double *u; double *item_u;
    /* method 64, several chains (pht_engine_set_chains): chains 0 .. chains-1, each with its own model block, stats block,
     * table and Philox key (ckeys[2c], ckeys[2c+1]) and observation counter cnext[c]; chain 0's blocks come first */
    /* method 64, groups (pht_engine_set_groups): unit u = c groups + g has model, stats and table block u and counter
     * cnext[u]; its layout positions are a kernel argument of the walker (pht_launch_unif).  `groups` sits in the padding
     * after `chains`, so the structure -- and the other kernels' code -- stays as it was. */
    int chains, groups; const uint32_t *ckeys; unsigned long long *cnext;
};

struct UpdateParams {
    double *model; long long *stats; DevState *state; double *res; int res_rows;
    const int *T; const double *C; const double *nu; const double *zeta;
    const int *var_ptr; const int *cell_i; const int *cell_j;   /* CSR: parameter -> cells in reference insertion order */
    int n, m, zbits; uint32_t k0, k1;
    const double *beta;        /* Dirichlet prior of the start distribution (n), nullptr: pi stays as it is */
    double *pires;             /* res_rows x n draws of pi, nullptr when pi is not inferred */
    /* several chains (method 64): one block of k_assemble / k_update / k_unif_table per chain; chain c's rows of res and
     * pires start at c x res_rows; ckeys as in SweepParams (nullptr: k0, k1); k_assemble zeroes cnext[c] when set */
    int chains; const uint32_t *ckeys; unsigned long long *cnext;
    /* groups (method 64): k_assemble and k_unif_table run one block per (chain, group) unit c groups + g, on T, C + g (n+1)^2
     * and the table span gtmax[g] (nullptr: the tmax argument); k_update (one block per chain) walks var_ptr[g m + v] ..
     * var_ptr[g m + v + 1] for g = 0 .. groups - 1 and writes theta and pi into every unit of its chain.  groups = 1 with
     * var_ptr of m + 1 entries is the single-structure engine. */
    int groups; const double *gtmax;
};

/* all-reduce of the statistics block through the exchange windows */
struct ReduceParams {
    long long *stats; int len; DevState *state;
    XchgWindow *xw; XchgWindow *xpeer[PHT_MAX_WORLD];
    uint32_t rank, world;
};

/* kernel launchers (each returns the cudaError of the launch) */
cudaError_t pht_launch_peer_allreduce(const ReduceParams &p, cudaStream_t st);
cudaError_t pht_launch_assemble(const UpdateParams &p, cudaStream_t st);
cudaError_t pht_launch_update(const UpdateParams &p, cudaStream_t st);
cudaError_t pht_launch_pack_error(const UpdateParams &p, cudaStream_t st);
cudaError_t pht_launch_mhrs(const SweepParams &p, int lane_blocks, int tail_blocks, int replay_blocks, cudaStream_t st);
/* mh: the LJMA_MHsample_Hobolth variant (method bit 8) instead of the live DCS sampler */
cudaError_t pht_launch_dcs(const SweepParams &p, int grid_blocks, cudaStream_t st, bool mh = false);
int pht_dcs_grid_blocks(int device, int n, bool mh = false);
/* ECS: exact and right-censored observations are separate launches over index lists (nullptr = identity) */
cudaError_t pht_launch_ecs(const SweepParams &p, int grid_blocks, const uint32_t *idx_exact, unsigned long long n_exact,
                           const uint32_t *idx_cens, unsigned long long n_cens, cudaStream_t st);
int pht_ecs_grid_blocks(int device, int n);
/* the LJMA_MHsample_Aslett variant (method bit 16): every observation of the list through the gt sampler + MH wrapper */
cudaError_t pht_launch_mhs_aslett(const SweepParams &p, int grid_blocks, const uint32_t *idx, unsigned long long count, cudaStream_t st);
int pht_mhs_aslett_grid_blocks(int device, int n);
/* spectral data of the sweep: inject != nullptr copies host-supplied (evals | Q | Qinv) instead of solving on the device */
cudaError_t pht_launch_spectral(const UpdateParams &p, const double *inject, cudaStream_t st);
/* iv: the instance that reads interval bounds (SweepParams::u != nullptr) */
int pht_mhrs_grid_blocks(int device, int n, bool iv, int *lane_blocks, int *tail_blocks, int *replay_blocks);
size_t pht_mhrs_smem_bytes(int n);
/* method 64 (k_unif.cu): log k! into a new table; the per-sweep table kernel (tmax: the longest time span of the shard,
 * max of y and of u - y); the path kernel and its grid.  The table (pht_unif.h, capacity PHT_UNIF_CAP powers) is a
 * kernel argument of its own, so that SweepParams / UpdateParams -- and the other kernels' code -- stay as they are. */
cudaError_t pht_unif_init(double *tab, int n, int cap, int chains, cudaStream_t st);   /* log k! of `chains` tables */
size_t pht_unif_table_doubles(int n, int cap);
cudaError_t pht_launch_unif_table(const UpdateParams &p, double *tab, double tmax, cudaStream_t st);
/* gofs: G + 1 offsets, group g's observations at layout positions [gofs[g], gofs[g + 1]) (nullptr: one group, [0, l_local)) */
cudaError_t pht_launch_unif(const SweepParams &p, const double *tab, const unsigned long long *gofs, int grid_blocks, cudaStream_t st);
int pht_unif_grid_blocks(int device, int n, bool chains);   /* chains: the kernel of several chains (k_unif_chain_paths) */
/* method 64, delayed entry (k_unif.cu; pht_engine_set_entry): a list of observations with entry ages and its buffers.
 * Like the table, every pointer is a kernel argument of its own. */
struct UnifEntry {
    const double *a; const uint32_t *obs; long first, count;   /* entry age per list entry; local observation index
                                                                  (obs == nullptr: first + i) */
    unsigned *M; unsigned long long *off;                      /* ghost counts and their exclusive scan, count + 1 each */
    double *etab; unsigned long long *next;                    /* sigma_k | phi_k (2 x PHT_UNIF_CAP); ghost hand-out counter */
    void *scan_tmp; size_t scan_bytes;                         /* CUB scratch of the scan */
    int count_blocks;                                          /* grid of the (grid-stride) count kernel at most */
};
#define PHT_ENTRY_COUNTS 1     /* entry tables, ghost counts, scan */
#define PHT_ENTRY_GHOSTS 2     /* the ghost paths */
cudaError_t pht_launch_unif_entry(const UpdateParams &u, const SweepParams &p, const double *tab, const UnifEntry &E, int ghost_blocks,
                                  int stages, cudaStream_t st);
size_t pht_unif_entry_scan_bytes(long count);
int pht_unif_ghost_grid_blocks(int device, int n);
/* large per-call buffers: stream-ordered pool allocations, cached across calls (engine.cu) */
cudaError_t pht_dev_alloc(void **p, size_t bytes, cudaStream_t st);
cudaError_t pht_dev_free(void *p, cudaStream_t st);
cudaError_t pht_sort_by_y_desc(const double *y, const uint8_t *cens, long l, double *ys, uint8_t *cs, uint32_t *perm, cudaStream_t st);
/* the grouped layout (pht_engine_set_groups): a stable radix sort by group id (ascending) of the y-descending permutation
 * perm_y (nullptr: the upload order), so each group is a contiguous range still ordered by decreasing y; group holds the
 * id of every local observation in upload order.  Writes perm, ys = y[perm], cs = cens[perm]. */
cudaError_t pht_sort_by_group(const uint32_t *perm_y, const uint8_t *group, const double *y, const uint8_t *cens, long l,
                              double *ys, uint8_t *cs, uint32_t *perm, cudaStream_t st);
/* dst[i] = src[perm[i]] (device arrays of length l) */
cudaError_t pht_gather_f64(const double *src, const uint32_t *perm, double *dst, long l, cudaStream_t st);

#endif
