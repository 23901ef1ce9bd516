/*
 * k_unif.cu -- the uniformisation path sampler (method 64) for sm_100a: exact conditional paths for any
 * sub-generator (Hobolth & Stone 2009, section 3.3), for exact, right-, interval- and left-censored observations.
 * Law, table, truncation and draw order: pht_unif.h, which this file and the host restatement share.
 *
 *   k_unif_lgk     once per engine (and per pht_engine_set_chains): log k! for k < capacity, in every chain's table
 *   k_unif_table   once per sweep (in place of k_spectral_solve): lambda, R = I + S/lambda, r = s/lambda and the
 *                  powers R^k, pi R^k, g_k for k <= K_sweep = K(lambda t_max), by sequential products.  One block per
 *                  chain: the products are a chain of K_sweep dependent steps, each n^2 + 2n dot products of length n, so
 *                  one step is one pass of the block over the entries with the previous power in shared memory.
 *   k_unif_paths   one observation per lane, persistent warps refilled from the global counter (Dispenser); the two
 *                  per-lane n-vectors of scratch live in shared-memory slabs (stride THREADS), the powers in global
 *                  memory (33 MB per chain at n = 32 and full capacity; what a sweep touches stays in L2).
 *   k_unif_chain_paths  the same per observation for several chains or groups: the blocks walk the (chain, group)
 *                  units (below)
 *
 * Delayed entry (only when entry ages are set, pht_engine_set_entry; law and draw order in pht_unif.h):
 *   k_unif_entry_table  sigma_k, phi_k for k <= K_sweep, after k_unif_table (one block)
 *   k_unif_entry_count  the ghost count M of every truncated observation, walked by decreasing a; then an exclusive
 *                       CUB scan of the counts (64-bit offsets) leaves the total G in device memory
 *   k_unif_ghosts       persistent warps over the flat ghost indices [0, G), one left-censored path per lane,
 *                       reduced into the same statistics block
 *
 * Counts (only when counts are set, pht_engine_set_counts; record form in pht_unif.h):
 *   k_unif_records      persistent warps over (chain, record chunk) items: a warp prepares the record's weights once
 *                       into its shared-memory slab, its lanes draw the chunk's units; records with few units run
 *                       through k_unif_paths / k_unif_chain_paths in an expanded layout of their own
 *
 * Bound: FP64 issue.  Per observation the sampler evaluates ~3 K(lambda y) Poisson weights (one pht_exp each) and
 * ~K(lambda y) n multiply-adds for the end-state weights, plus n per uniformised event; the observations are handed out
 * by decreasing y (k_sort.cu), so the lanes of a warp run similar K.
 */
#include <cub/device/device_scan.cuh>
#include <cuda/std/functional>
#include "path_common.cuh"

/* one out-of-line uniform: the sampler draws at a dozen places of a divergent body */
static __device__ __noinline__ double unif_u01(pht_stream *st) { return pht_stream_unif(st); }
struct UnifCount { const SweepParams *p; unsigned int *Nacc; long out_idx; int n; };
#define PHT_UNIF_U01(st) unif_u01(st)
#define PHT_UNIF_FN static __device__ __forceinline__
#define PHT_UNIF_CTX UnifCount
#define PHT_UNIF_COUNT(ctx, from, to) count_transition(*(ctx)->p, (ctx)->n, (ctx)->Nacc, (ctx)->out_idx, (from), (to))
#include "pht_unif.h"

#define UNIF_THREADS 128
#define UNIF_TABLE_THREADS 256

/* block c fills table c */
__global__ void k_unif_lgk(double *tab, int n, int cap) {
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    if (threadIdx.x == 0) pht_unif_lgk_fill(tab + (size_t)blockIdx.x * L.total + L.lgk, cap);
}

/* block c builds unit c's table from unit c's model block (grid = chains x groups); a group's table spans its own
 * observations (gtmax[c % groups]): a path never reads a power beyond its own K(lambda y), so the span changes no bit */
__global__ void __launch_bounds__(UNIF_TABLE_THREADS) k_unif_table(UpdateParams p, double *tab, double tmax) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = p.n, nn = n * n, tid = threadIdx.x, cap = PHT_UNIF_CAP;
    const ModelLayout ML = ModelLayout::make(n, p.m);
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    const double *model = p.model + (size_t)blockIdx.x * ML.total;
    tab += (size_t)blockIdx.x * L.total;
    const double *S = model + ML.S, *s = model + ML.s, *pi = model + ML.pi;
    double *sR = reinterpret_cast<double *>(smem_raw), *sr = sR + nn;
    double *P0 = sr + n, *P1 = P0 + nn, *q0 = P1 + nn, *q1 = q0 + n, *g0 = q1 + n, *g1 = g0 + n;
    const double lam = pht_unif_lambda(n, S);
    if (p.gtmax) tmax = p.gtmax[blockIdx.x % p.groups];
    int K = pht_unif_K(lam * tmax);
    if (K >= cap) { if (tid == 0) atomicOr(&p.state->error, PHT_UNIF_ERR_TABLE); K = cap - 1; }
    for (int e = tid; e < nn; e += blockDim.x) {
        const double v = pht_unif_R_entry(n, S, lam, e % n, e / n);
        sR[e] = v; tab[L.R + e] = v;
        P0[e] = (e % n == e / n) ? 1.0 : 0.0; tab[L.P + e] = P0[e];
    }
    for (int i = tid; i < n; i += blockDim.x) {
        const double v = s[i] / lam;
        sr[i] = v; tab[L.r + i] = v;
        q0[i] = pi[i]; tab[L.q + i] = pi[i];
        g0[i] = 0.0; tab[L.g + i] = 0.0;
    }
    if (tid == 0) {
        int npos = 0, a1 = 0;
        for (int i = n - 1; i >= 0; i--) if (pi[i] > 0.0) { npos++; a1 = i; }
        tab[0] = lam; tab[1] = K; tab[2] = npos; tab[3] = a1;
    }
    for (int k = 0; k < K; k++) {
        __syncthreads();
        double *Pn = tab + L.P + (k + 1) * nn, *qn = tab + L.q + (k + 1) * n, *gn = tab + L.g + (k + 1) * n;
        for (int e = tid; e < nn + 2 * n; e += blockDim.x) {
            if (e < nn) { const double v = pht_unif_P_entry(n, P0, sR, e % n, e / n); P1[e] = v; Pn[e] = v; }
            else if (e < nn + n) { const int j = e - nn; const double v = pht_unif_q_entry(n, q0, sR, j); q1[j] = v; qn[j] = v; }
            else { const int i = e - nn - n; const double v = pht_unif_g_entry(n, g0, sR, sr, i); g1[i] = v; gn[i] = v; }
        }
        double *t;
        t = P0; P0 = P1; P1 = t; t = q0; q0 = q1; q1 = t; t = g0; g0 = g1; g1 = t;
    }
}

template <int THREADS>
struct UnifSmem {
    double *Za, *Zb, *s, *scale, *cum, *pi;
    unsigned long long *zlo; long long *zhi; unsigned int *Nacc, *Bacc;
    __device__ __forceinline__ void carve(unsigned char *raw, int n) {
        double *d = reinterpret_cast<double *>(raw);
        Za = d; d += n * THREADS; Zb = d; d += n * THREADS;
        s = d; d += n; scale = d; d += n; cum = d; d += (n + 1) * (n + 1); pi = d; d += n;
        zlo = reinterpret_cast<unsigned long long *>(d); d += n; zhi = reinterpret_cast<long long *>(d); d += n;
        Nacc = reinterpret_cast<unsigned int *>(d); Bacc = Nacc + n * n;
    }
    static size_t bytes(int n) {
        return sizeof(double) * (size_t)(2 * n * THREADS + 3 * n + (n + 1) * (n + 1) + 2 * n) + sizeof(unsigned int) * (size_t)(n * n + n);
    }
};

template <int THREADS>
__global__ void __launch_bounds__(THREADS) k_unif_paths(SweepParams p, const double *tab) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = p.n, tid = threadIdx.x;
    const unsigned FULL = 0xffffffffu;
    const ModelLayout ML = ModelLayout::make(n, p.m);
    UnifSmem<THREADS> sm; sm.carve(smem_raw, n);
    for (int i = tid; i < n * n; i += THREADS) sm.Nacc[i] = 0u;
    for (int i = tid; i < (n + 1) * (n + 1); i += THREADS) sm.cum[i] = p.model[ML.cum + i];
    for (int i = tid; i < n; i += THREADS) {
        sm.s[i] = p.model[ML.s + i]; sm.scale[i] = p.model[ML.scale + i]; sm.pi[i] = p.model[ML.pi + i];
        sm.zlo[i] = 0ull; sm.zhi[i] = 0; sm.Bacc[i] = 0u;
    }
    __syncthreads();
    const uint32_t iter = p.state->iter;
    unsigned c_paths = 0; int err = 0;
    Dispenser disp; disp.init(p);
    UnifCount ctx; ctx.p = &p; ctx.Nacc = sm.Nacc; ctx.n = n; ctx.out_idx = 0;
    for (;;) {
        const unsigned long long o = disp.take(p, FULL, true);
        const bool have = o != ~0ull;
        if (__ballot_sync(FULL, have) == 0u) { if (disp.exhausted) break; continue; }
        if (have) {
            const uint32_t obs_local = p.perm ? p.perm[o] : (uint32_t)o;
            pht_stream st; st.k0 = p.k0; st.k1 = p.k1;
            pht_stream_seek(&st, iter, p.obs_rank + obs_local * p.obs_world, 0u, 0u);
            ctx.out_idx = (long)o - p.first;
            int B = 0;
            err |= pht_unif_path(tab, n, PHT_UNIF_CAP, sm.s, sm.scale, sm.cum, sm.pi, p.y[o], p.cens[o],
                                 p.u ? p.u[o] : INFINITY, &st, sm.Za + tid, sm.Zb + tid, THREADS, &ctx, &B);
            path_flush<THREADS>(p, n, sm.Za, sm.zlo, sm.zhi, sm.Bacc, B, ctx.out_idx);
            c_paths++;
        }
        __syncwarp();
    }
    if (err) atomicOr(&p.state->error, err);
    __syncthreads();
    block_flush<THREADS>(p, n, sm.Nacc, sm.Bacc, sm.zlo, sm.zhi);
    unsigned long long w_paths = c_paths;
    for (int o = 16; o > 0; o >>= 1) w_paths += __shfl_down_sync(FULL, w_paths, o);
    if ((tid & 31) == 0) atomicAdd(&p.state->counters[PHT_CNT_PATHS], w_paths);
}

/* Several chains or groups (pht_engine_set_chains, pht_engine_set_groups; one chain of one group and parity mode run
 * k_unif_paths above, 2 % faster at one chain on the C3 shape).  The work comes in units u = c groups + g: chain c's paths
 * of group g's observations, layout positions [gofs[g], gofs[g + 1]), drawn with chain c's key on unit u's model and
 * table into unit u's statistics block, handed out by unit u's counter.  Persistent blocks walk the units: block b starts
 * at unit b mod units, loads that unit's model into shared memory and its warps take observations 32 at a time from the
 * unit's counter.  When the counter runs dry the block flushes its accumulators into the unit's statistics block and
 * moves on to the next unit that still has work, until it has passed every unit once.  Whether a unit has work left is
 * read from its counter with plain loads, 32 units per warp-wide look; every statistic is an integer sum, so which block
 * draws which observation does not change the result. */
template <int THREADS>
__global__ void __launch_bounds__(THREADS, 7) /* 7 blocks of 128 per SM: at most 72 registers */ k_unif_chain_paths(SweepParams p, const double *tab,
                                                                                                             const unsigned long long *gofs) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    /* the walk's state lives in shared memory, re-read after each barrier, so that it holds no register in the path loop */
    __shared__ int s_chain, s_left; __shared__ uint32_t s_key[2];
    __shared__ const double *s_tab; __shared__ unsigned long long *s_counter, s_begin, s_end;
    const int n = p.n, tid = threadIdx.x;
    const unsigned FULL = 0xffffffffu;
    const ModelLayout ML = ModelLayout::make(n, p.m);
    const int chains = p.chains * p.groups;       /* units (s_chain: the current one) */
    UnifSmem<THREADS> sm; sm.carve(smem_raw, n);
    const uint32_t iter = p.state->iter;
    unsigned c_paths = 0; int err = 0;
    Dispenser disp; disp.init(p);
    UnifCount ctx; ctx.p = &p; ctx.Nacc = sm.Nacc; ctx.n = n; ctx.out_idx = 0;
    if (tid == 0) { s_chain = (int)(blockIdx.x % (unsigned)chains); s_left = chains; }   /* current chain; chains not passed yet */
    __syncthreads();
    for (;;) {
        if (tid < 32) {                        /* the first chain from the current one on (cyclically) with work left */
            const int c = s_chain, left = s_left;
            int found = -1;
            for (int k = 0; k < left && found < 0; k += 32) {
                int cc = c + k + tid; if (cc >= chains) cc -= chains;
                const int g = cc % p.groups;
                const unsigned long long span = gofs ? gofs[g + 1] - gofs[g] : (unsigned long long)p.l_local;
                const bool work = k + tid < left && *(volatile unsigned long long *)&p.cnext[cc] < span;
                const unsigned b = __ballot_sync(FULL, work);
                if (b) found = k + __ffs(b) - 1;
            }
            if (tid == 0) {
                int cn = c + (found < 0 ? 0 : found); if (cn >= chains) cn -= chains;
                s_chain = cn; s_left = found < 0 ? 0 : left - found;
                const int ch = cn / p.groups, g = cn - ch * p.groups;
                s_key[0] = p.ckeys[2 * ch]; s_key[1] = p.ckeys[2 * ch + 1];
                s_tab = tab + (size_t)cn * pht_unif_layout_make(n, PHT_UNIF_CAP).total; s_counter = p.cnext + cn;
                s_begin = gofs ? gofs[g] : 0ull; s_end = gofs ? gofs[g + 1] : (unsigned long long)p.l_local;
            }
        }
        __syncthreads();
        if (s_left == 0) break;
        {
            const double *model = p.model + (size_t)s_chain * ML.total;
            for (int i = tid; i < n * n; i += THREADS) sm.Nacc[i] = 0u;
            for (int i = tid; i < (n + 1) * (n + 1); i += THREADS) sm.cum[i] = model[ML.cum + i];
            for (int i = tid; i < n; i += THREADS) {
                sm.s[i] = model[ML.s + i]; sm.scale[i] = model[ML.scale + i]; sm.pi[i] = model[ML.pi + i];
                sm.zlo[i] = 0ull; sm.zhi[i] = 0; sm.Bacc[i] = 0u;
            }
        }
        __syncthreads();
        disp.next = disp.end = 0ull; disp.exhausted = false; disp.obs_begin = s_begin; disp.obs_end = s_end;
        for (;;) {
            const unsigned long long o = disp.take_from(s_counter, FULL, true);
            const bool have = o != ~0ull;
            if (__ballot_sync(FULL, have) == 0u) { if (disp.exhausted) break; continue; }
            if (have) {
                const uint32_t obs_local = p.perm ? p.perm[o] : (uint32_t)o;
                pht_stream st; st.k0 = s_key[0]; st.k1 = s_key[1];
                pht_stream_seek(&st, iter, p.obs_rank + obs_local * p.obs_world, 0u, 0u);
                ctx.out_idx = (long)o - p.first;
                int B = 0;
                err |= pht_unif_path(s_tab, n, PHT_UNIF_CAP, sm.s, sm.scale, sm.cum, sm.pi, p.y[o], p.cens[o],
                                     p.u ? p.u[o] : INFINITY, &st, sm.Za + tid, sm.Zb + tid, THREADS, &ctx, &B);
                path_flush<THREADS>(p, n, sm.Za, sm.zlo, sm.zhi, sm.Bacc, B, ctx.out_idx);
                c_paths++;
            }
            __syncwarp();
        }
        __syncthreads();
        block_flush_to<THREADS>(p.stats + (size_t)s_chain * stats_len(n), n, sm.Nacc, sm.Bacc, sm.zlo, sm.zhi);
        __syncthreads();
        if (tid == 0) { int cn = s_chain + 1; if (cn == chains) cn = 0; s_chain = cn; s_left = s_left - 1; }
        __syncthreads();
    }
    if (err) atomicOr(&p.state->error, err);
    unsigned long long w_paths = c_paths;
    for (int o = 16; o > 0; o >>= 1) w_paths += __shfl_down_sync(FULL, w_paths, o);
    if ((tid & 31) == 0) atomicAdd(&p.state->counters[PHT_CNT_PATHS], w_paths);
}

/* ---- delayed entry (pht_unif.h, "Delayed entry"): launched only when entry ages are set */

/* sigma_k and phi_k for k <= K_sweep, after k_unif_table; one block */
__global__ void __launch_bounds__(UNIF_TABLE_THREADS) k_unif_entry_table(UpdateParams p, const double *tab, double *etab) {
    const int n = p.n, cap = PHT_UNIF_CAP;
    const ModelLayout ML = ModelLayout::make(n, p.m);
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    const double *pi = p.model + ML.pi;
    const int K = (int)tab[1];
    for (int k = threadIdx.x; k <= K; k += blockDim.x) {
        etab[k] = pht_unif_sigma_entry(n, tab + L.q + k * n);
        etab[cap + k] = pht_unif_phi_entry(n, pi, tab + L.g + k * n);
    }
}

/* the ghost count of every entry of a list (a[i], local observation obs[i], or first + i when obs is null); M[count] = 0
 * closes the list for the scan */
__global__ void __launch_bounds__(256) k_unif_entry_count(SweepParams p, const double *tab, const double *etab, const double *a,
                                                        const uint32_t *obs, long first, long count, unsigned *M) {
    const uint32_t iter = p.state->iter;
    int err = 0;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i <= count; i += (long)gridDim.x * blockDim.x) {
        unsigned m = 0u;
        if (i < count && a[i] > 0.0) {
            const uint32_t ol = obs ? obs[i] : (uint32_t)(first + i);
            const double U = pht_unif_at(p.k0, p.k1, iter, p.obs_rank + ol * p.obs_world, 1u, 0u);
            err |= pht_unif_ghost_count(tab, etab, p.n, PHT_UNIF_CAP, a[i], U, &m);
        }
        M[i] = m;
    }
    if (err) atomicOr(&p.state->error, err);
}

/* Ghost paths.  Persistent warps take 32 flat ghost indices g in [0, G) at a time (G = off[count], on the device) and
 * map each to (list entry i, ghost j): a binary search for the chunk's first index, then per lane a galloping search
 * from there over the entries with no ghosts.  Each lane runs the shared sampler (y = 0, censored, u = a on sub-stream
 * 2 + j) and reduces the path into the sweep statistics like k_unif_paths; in parity mode (p.outB) ghost g is record g. */
template <int THREADS>
__global__ void __launch_bounds__(THREADS) k_unif_ghosts(SweepParams p, const double *tab, const double *a, const uint32_t *obs,
                                                         long first, long count, const unsigned long long *off,
                                                         unsigned long long *next) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = p.n, tid = threadIdx.x, lane = tid & 31;
    const unsigned FULL = 0xffffffffu;
    const ModelLayout ML = ModelLayout::make(n, p.m);
    UnifSmem<THREADS> sm; sm.carve(smem_raw, n);
    for (int i = tid; i < n * n; i += THREADS) sm.Nacc[i] = 0u;
    for (int i = tid; i < (n + 1) * (n + 1); i += THREADS) sm.cum[i] = p.model[ML.cum + i];
    for (int i = tid; i < n; i += THREADS) {
        sm.s[i] = p.model[ML.s + i]; sm.scale[i] = p.model[ML.scale + i]; sm.pi[i] = p.model[ML.pi + i];
        sm.zlo[i] = 0ull; sm.zhi[i] = 0; sm.Bacc[i] = 0u;
    }
    __syncthreads();
    const uint32_t iter = p.state->iter;
    const unsigned long long G = off[count];
    int err = 0;
    UnifCount ctx; ctx.p = &p; ctx.Nacc = sm.Nacc; ctx.n = n; ctx.out_idx = 0;
    for (;;) {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(next, (unsigned long long)PATH_CHUNK);
        base = __shfl_sync(FULL, base, 0);
        if (base >= G) break;
        long lo = 0, hi = count;                       /* the entry holding ghost `base`: off[lo] <= base < off[lo + 1] */
        while (hi - lo > 1) { const long mid = (lo + hi) >> 1; if (off[mid] <= base) lo = mid; else hi = mid; }
        const unsigned long long g = base + (unsigned long long)lane;
        if (g < G) {
            long i = lo;
            if (off[i + 1] <= g) {                     /* off[count] = G > g bounds the search */
                long l0 = i, h0 = i, step = 1;
                for (;;) {
                    h0 = i + step;
                    if (h0 >= count - 1) { h0 = count - 1; break; }
                    if (off[h0 + 1] > g) break;
                    l0 = h0; step <<= 1;
                }
                while (h0 - l0 > 1) { const long mid = (l0 + h0) >> 1; if (off[mid + 1] > g) h0 = mid; else l0 = mid; }
                i = h0;
            }
            const uint32_t ol = obs ? obs[i] : (uint32_t)(first + i);
            pht_stream st; st.k0 = p.k0; st.k1 = p.k1;
            pht_stream_seek(&st, iter, p.obs_rank + ol * p.obs_world, 2u + (uint32_t)(g - off[i]), 0u);
            ctx.out_idx = (long)g;
            int B = 0;
            err |= pht_unif_path(tab, n, PHT_UNIF_CAP, sm.s, sm.scale, sm.cum, sm.pi, 0.0, 1, a[i], &st,
                                 sm.Za + tid, sm.Zb + tid, THREADS, &ctx, &B);
            path_flush<THREADS>(p, n, sm.Za, sm.zlo, sm.zhi, sm.Bacc, B, ctx.out_idx);
        }
        __syncwarp();
    }
    if (err) atomicOr(&p.state->error, err);
    __syncthreads();
    block_flush<THREADS>(p, n, sm.Nacc, sm.Bacc, sm.zlo, sm.zhi);
}

/* ---- records with counts (pht_engine_set_counts; pht_unif.h, "Records with counts"): launched only when counts are set.
 * Work items are (record, chunk of at most PHT_COUNTS_CHUNK units) of the records at or above the count threshold; the
 * hand-out runs over (chain, item), unit = c groups + item's group as in k_unif_chain_paths.  A persistent warp takes one
 * work item at a time, prepares the record into its shared-memory slab (lanes over k for the weights, over states and
 * cells for the vector and the matrix), then its lanes draw the chunk's units, one per lane, 32 at a time, into the
 * warp's own accumulators, which are flushed into the unit's statistics block after every item (so no 32-bit counter
 * can wrap, whatever the count).  Unit j of record k is expanded observation base_k + j: Philox sub-stream 0 of (sweep,
 * base_k + j) with chain c's key. */
#define UNIF_REC_KB 255              /* weights a slab holds per record (k = 0 .. KB); beyond, pht_unif_w recomputes them */

struct UnifRecSlab {
    double *w1, *w2, *v, *mx; unsigned long long *zlo; long long *zhi; unsigned int *Nacc, *Bacc;
    __host__ __device__ static size_t bytes(int n) {
        return sizeof(double) * (size_t)(2 * (UNIF_REC_KB + 1) + n + n * n + 2 * n) + sizeof(unsigned int) * (size_t)(n * n + n);
    }
    __device__ __forceinline__ void carve(unsigned char *raw, int n) {
        double *d = reinterpret_cast<double *>(raw);
        w1 = d; d += UNIF_REC_KB + 1; w2 = d; d += UNIF_REC_KB + 1; v = d; d += n; mx = d; d += n * n;
        zlo = reinterpret_cast<unsigned long long *>(d); d += n; zhi = reinterpret_cast<long long *>(d); d += n;
        Nacc = reinterpret_cast<unsigned int *>(d); Bacc = Nacc + n * n;
    }
};
template <int THREADS>
static size_t unif_rec_smem(int n) {       /* per-lane path scratch (stride THREADS) + one slab per warp, 16-byte aligned */
    return sizeof(double) * (size_t)(2 * n * THREADS) + (size_t)(THREADS / 32) * ((UnifRecSlab::bytes(n) + 15) & ~(size_t)15);
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS) k_unif_records(SweepParams p, const double *tab, UnifRecords R) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = p.n, tid = threadIdx.x, lane = tid & 31, cap = PHT_UNIF_CAP;
    const unsigned FULL = 0xffffffffu;
    const ModelLayout ML = ModelLayout::make(n, p.m);
    const pht_unif_layout TL = pht_unif_layout_make(n, cap);
    double *Za = reinterpret_cast<double *>(smem_raw), *Zb = Za + n * THREADS;
    UnifRecSlab w;
    w.carve(smem_raw + sizeof(double) * (size_t)(2 * n * THREADS) + (size_t)(tid >> 5) * ((UnifRecSlab::bytes(n) + 15) & ~(size_t)15), n);
    for (int i = lane; i < n * n; i += 32) w.Nacc[i] = 0u;
    for (int i = lane; i < n; i += 32) { w.Bacc[i] = 0u; w.zlo[i] = 0ull; w.zhi[i] = 0; }
    __syncwarp();
    const uint32_t iter = p.state->iter;
    const unsigned long long work = (unsigned long long)p.chains * (unsigned long long)R.n_items;
    unsigned long long c_paths = 0; int err = 0;
    UnifCount ctx; ctx.p = &p; ctx.Nacc = w.Nacc; ctx.n = n; ctx.out_idx = 0;
    for (;;) {
        unsigned long long f = 0;
        if (lane == 0) f = atomicAdd(R.next, 1ull);
        f = __shfl_sync(FULL, f, 0);
        if (f >= work) break;
        const unsigned c = (unsigned)(f / (unsigned long long)R.n_items);
        const uint4 it = R.items[f - (unsigned long long)c * R.n_items];       /* record, first unit, units, group */
        const int unit = (int)c * p.groups + (int)it.w;
        const double *utab = tab + (size_t)unit * TL.total, *model = p.model + (size_t)unit * ML.total;
        pht_unif_rec rc;
        const int e0 = pht_unif_rec_init(&rc, utab, cap, R.y[it.x], R.cens[it.x], R.u ? R.u[it.x] : INFINITY, UNIF_REC_KB);
        if (e0) { err |= e0; continue; }
        rc.w1 = w.w1; rc.w2 = w.w2; rc.v = w.v; rc.mx = w.mx;
        const double *lgk = utab + TL.lgk;
        const int k1 = rc.K1 < UNIF_REC_KB ? rc.K1 : UNIF_REC_KB, k2 = !rc.iv ? -1 : rc.K2 < UNIF_REC_KB ? rc.K2 : UNIF_REC_KB;
        for (int k = lane; k <= k1; k += 32) w.w1[k] = pht_unif_w(rc.x, rc.lx, k, lgk);
        for (int k = lane; k <= k2; k += 32) w.w2[k] = pht_unif_w(rc.x2, rc.lx2, k, lgk);
        __syncwarp();
        if (lane < n) w.v[lane] = pht_unif_rec_v_entry(&rc, utab, n, cap, model + ML.s, lane);
        if (rc.y > 0.0 && (int)utab[2] > 1)
            for (int e = lane; e < n * n; e += 32) w.mx[e] = pht_unif_rec_m_entry(&rc, utab, n, cap, model + ML.pi, e % n, e / n);
        __syncwarp();
        const uint32_t k0 = p.ckeys[2 * c], k1key = p.ckeys[2 * c + 1], base = R.base[it.x] + it.y;
        for (unsigned j = lane; j < it.z; j += 32) {
            pht_stream st; st.k0 = k0; st.k1 = k1key;
            pht_stream_seek(&st, iter, base + j, 0u, 0u);
            int B = 0;
            err |= pht_unif_rec_path(utab, n, cap, model + ML.scale, model + ML.cum, &rc, &st, Za + tid, Zb + tid, THREADS, &ctx, &B);
            path_flush<THREADS>(p, n, Za, w.zlo, w.zhi, w.Bacc, B, 0);
            c_paths++;
        }
        __syncwarp();
        unsigned long long *g = reinterpret_cast<unsigned long long *>(p.stats + (size_t)unit * stats_len(n));
        for (int i = lane; i < n * n; i += 32) if (w.Nacc[i]) { atomicAdd(&g[i], (unsigned long long)w.Nacc[i]); w.Nacc[i] = 0u; }
        for (int i = lane; i < n; i += 32) {
            if (w.Bacc[i]) { atomicAdd(&g[n * n + i], (unsigned long long)w.Bacc[i]); w.Bacc[i] = 0u; }
            if (w.zlo[i]) { atomicAdd(&g[n * n + n + i], w.zlo[i]); w.zlo[i] = 0ull; }
            if (w.zhi[i]) { atomicAdd(&g[n * n + 2 * n + i], (unsigned long long)w.zhi[i]); w.zhi[i] = 0; }
        }
        __syncwarp();
    }
    if (err) atomicOr(&p.state->error, err);
    for (int o = 16; o > 0; o >>= 1) c_paths += __shfl_down_sync(FULL, c_paths, o);
    if (lane == 0) atomicAdd(&p.state->counters[PHT_CNT_PATHS], c_paths);
}

int pht_unif_records_grid_blocks(int device, int n) {
    const size_t smem = unif_rec_smem<UNIF_THREADS>(n);
    int per_sm = 0, sms = 0;
    if (cudaFuncSetAttribute(k_unif_records<UNIF_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_unif_records<UNIF_THREADS>, UNIF_THREADS, smem) != cudaSuccess) return -1;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return -1;
    return per_sm * sms;
}

cudaError_t pht_launch_unif_records(const SweepParams &p, const double *tab, const UnifRecords &R, int grid_blocks, cudaStream_t st) {
    const cudaError_t e = cudaMemsetAsync(R.next, 0, sizeof(unsigned long long), st);
    if (e != cudaSuccess) return e;
    k_unif_records<UNIF_THREADS><<<grid_blocks, UNIF_THREADS, unif_rec_smem<UNIF_THREADS>(p.n), st>>>(p, tab, R);
    return cudaGetLastError();
}

/* ---- panel observations (pht_engine_set_visits; pht_unif.h, "Panel observations"): launched only when some observation
 * has visits, over those observations alone (the others run through k_unif_paths / k_unif_chain_paths in a layout of their
 * own).  Work items are (chain, chunk of at most 32 panel observations of one group), chunk r of chain c at flat index
 * c chunks + r, so every item belongs to one unit c groups + g.  A persistent warp takes one item at a time; its lanes draw
 * one observation each (model and table of the unit from global memory) into the warp's own accumulators, which are
 * flushed into the unit's statistics block after every item.  The lanes' n-vectors of path scratch live in shared-memory
 * slabs as in k_unif_paths; the beta history, (visits + 1) n doubles per observation, in global scratch, one slot per
 * resident lane (stride: the grid's lanes, so a warp's lanes touch adjacent words). */
struct UnifPanelAcc {
    unsigned long long *zlo; long long *zhi; unsigned int *Nacc, *Bacc;
    __host__ __device__ static size_t bytes(int n) { return sizeof(double) * (size_t)(2 * n) + sizeof(unsigned int) * (size_t)(n * n + n); }
    __device__ __forceinline__ void carve(unsigned char *raw, int n) {
        zlo = reinterpret_cast<unsigned long long *>(raw); zhi = reinterpret_cast<long long *>(zlo + n);
        Nacc = reinterpret_cast<unsigned int *>(zhi + n); Bacc = Nacc + n * n;
    }
};
template <int THREADS>
static size_t unif_panel_smem(int n) {     /* per-lane path scratch (stride THREADS) + one accumulator set per warp, 16-byte aligned */
    return sizeof(double) * (size_t)(2 * n * THREADS) + (size_t)(THREADS / 32) * ((UnifPanelAcc::bytes(n) + 15) & ~(size_t)15);
}

/* twin: k_unif_emis_paths below repeats this kernel for stage visits; a fix to one belongs in the other */
template <int THREADS>
__global__ void __launch_bounds__(THREADS) k_unif_panel_paths(SweepParams p, const double *tab, UnifPanel V) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = p.n, tid = threadIdx.x, lane = tid & 31, cap = PHT_UNIF_CAP, G = p.groups;
    const unsigned FULL = 0xffffffffu;
    const ModelLayout ML = ModelLayout::make(n, p.m);
    const size_t tabd = (size_t)pht_unif_layout_make(n, cap).total;
    double *Za = reinterpret_cast<double *>(smem_raw), *Zb = Za + n * THREADS;
    UnifPanelAcc w;
    w.carve(smem_raw + sizeof(double) * (size_t)(2 * n * THREADS) + (size_t)(tid >> 5) * ((UnifPanelAcc::bytes(n) + 15) & ~(size_t)15), n);
    for (int i = lane; i < n * n; i += 32) w.Nacc[i] = 0u;
    for (int i = lane; i < n; i += 32) { w.Bacc[i] = 0u; w.zlo[i] = 0ull; w.zhi[i] = 0; }
    __syncwarp();
    const uint32_t iter = p.state->iter;
    const long bs = (long)gridDim.x * THREADS;
    double *beta = V.beta + (size_t)blockIdx.x * THREADS + tid;
    const unsigned long long chunks = V.coff[G], work = (unsigned long long)p.chains * chunks;
    unsigned long long c_paths = 0; int err = 0;
    UnifCount ctx; ctx.p = &p; ctx.Nacc = w.Nacc; ctx.n = n; ctx.out_idx = 0;
    for (;;) {
        unsigned long long f = 0;
        if (lane == 0) f = atomicAdd(V.next, 1ull);
        f = __shfl_sync(FULL, f, 0);
        if (f >= work) break;
        const unsigned c = (unsigned)(f / chunks);
        const unsigned long long r = f - (unsigned long long)c * chunks;
        int g = 0;
        while (V.coff[g + 1] <= r) g++;
        const unsigned long long j0 = V.gofs[g] + (r - V.coff[g]) * 32ull, j = j0 + (unsigned long long)lane;
        const int unit = (int)c * G + g;
        const double *utab = tab + (size_t)unit * tabd, *model = p.model + (size_t)unit * ML.total;
        if (j < V.gofs[g + 1]) {
            const uint32_t ol = V.perm[j];
            pht_stream st; st.k0 = p.ckeys[2 * c]; st.k1 = p.ckeys[2 * c + 1];
            pht_stream_seek(&st, iter, p.obs_rank + ol * p.obs_world, 0u, 0u);
            ctx.out_idx = (long)ol - p.first;
            const unsigned long long v0 = V.voff[j];
            int B = 0;
            err |= pht_unif_panel_path(utab, n, cap, model + ML.s, model + ML.scale, model + ML.cum, model + ML.pi, V.y[j], V.cens[j],
                                       V.u ? V.u[j] : INFINITY, (int)(V.voff[j + 1] - v0), V.vt + v0, V.vm + v0, beta, bs, &st,
                                       Za + tid, Zb + tid, THREADS, &ctx, &B);
            path_flush<THREADS>(p, n, Za, w.zlo, w.zhi, w.Bacc, B, ctx.out_idx);
            c_paths++;
        }
        __syncwarp();
        if (p.outB == nullptr) {
            unsigned long long *gs = reinterpret_cast<unsigned long long *>(p.stats + (size_t)unit * stats_len(n));
            for (int i = lane; i < n * n; i += 32) if (w.Nacc[i]) { atomicAdd(&gs[i], (unsigned long long)w.Nacc[i]); w.Nacc[i] = 0u; }
            for (int i = lane; i < n; i += 32) {
                if (w.Bacc[i]) { atomicAdd(&gs[n * n + i], (unsigned long long)w.Bacc[i]); w.Bacc[i] = 0u; }
                if (w.zlo[i]) { atomicAdd(&gs[n * n + n + i], w.zlo[i]); w.zlo[i] = 0ull; }
                if (w.zhi[i]) { atomicAdd(&gs[n * n + 2 * n + i], (unsigned long long)w.zhi[i]); w.zhi[i] = 0; }
            }
        }
        __syncwarp();
    }
    if (err) atomicOr(&p.state->error, err);
    for (int o = 16; o > 0; o >>= 1) c_paths += __shfl_down_sync(FULL, c_paths, o);
    if (lane == 0) atomicAdd(&p.state->counters[PHT_CNT_PATHS], c_paths);
}

int pht_unif_panel_grid_blocks(int device, int n) {
    const size_t smem = unif_panel_smem<PHT_UNIF_PANEL_THREADS>(n);
    int per_sm = 0, sms = 0;
    if (cudaFuncSetAttribute(k_unif_panel_paths<PHT_UNIF_PANEL_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_unif_panel_paths<PHT_UNIF_PANEL_THREADS>, PHT_UNIF_PANEL_THREADS, smem) != cudaSuccess) return -1;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return -1;
    return per_sm * sms;
}

cudaError_t pht_launch_unif_panel(const SweepParams &p, const double *tab, const UnifPanel &V, int grid_blocks, cudaStream_t st) {
    const cudaError_t e = cudaMemsetAsync(V.next, 0, sizeof(unsigned long long), st);
    if (e != cudaSuccess) return e;
    k_unif_panel_paths<PHT_UNIF_PANEL_THREADS><<<grid_blocks, PHT_UNIF_PANEL_THREADS, unif_panel_smem<PHT_UNIF_PANEL_THREADS>(p.n), st>>>(p, tab, V);
    return cudaGetLastError();
}

/* ---- misclassified panel observations (pht_engine_set_stage_visits; pht_unif.h, "Misclassified panel observations"):
 * k_unif_panel_paths with stage indices in V.vm and the emission matrix of the item's chain, drawn by pht_unif_emis_path.
 * Besides the statistics, every warp counts its lanes' visits by (drawn phase, stage read) in n S shared-memory counters
 * of its own, flushed into the chain's 64-bit K block after every item, as the statistics are.  Counted only when the
 * statistics are (p.outB nullptr). */
template <int THREADS>
static size_t unif_emis_smem(int n, int S) {
    return unif_panel_smem<THREADS>(n) + (size_t)(THREADS / 32) * sizeof(unsigned int) * (size_t)(n * S);
}

/* twin of k_unif_panel_paths above (kept apart so that its SASS stays as it is); a fix to one belongs in the other.  The
 * minimum of 4 blocks lets ptxas use the registers it needs: without it, it settles on 72 registers and spills */
template <int THREADS>
__global__ void __launch_bounds__(THREADS, 4) k_unif_emis_paths(SweepParams p, const double *tab, UnifPanel V, UnifEmis X) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = p.n, tid = threadIdx.x, lane = tid & 31, cap = PHT_UNIF_CAP, G = p.groups, S = X.S, nS = n * S;
    const unsigned FULL = 0xffffffffu;
    const ModelLayout ML = ModelLayout::make(n, p.m);
    const size_t tabd = (size_t)pht_unif_layout_make(n, cap).total;
    double *Za = reinterpret_cast<double *>(smem_raw), *Zb = Za + n * THREADS;
    UnifPanelAcc w;
    w.carve(smem_raw + sizeof(double) * (size_t)(2 * n * THREADS) + (size_t)(tid >> 5) * ((UnifPanelAcc::bytes(n) + 15) & ~(size_t)15), n);
    unsigned int *Kacc = reinterpret_cast<unsigned int *>(smem_raw + sizeof(double) * (size_t)(2 * n * THREADS)
                                                          + (size_t)(THREADS / 32) * ((UnifPanelAcc::bytes(n) + 15) & ~(size_t)15)) + (size_t)(tid >> 5) * nS;
    for (int i = lane; i < n * n; i += 32) w.Nacc[i] = 0u;
    for (int i = lane; i < n; i += 32) { w.Bacc[i] = 0u; w.zlo[i] = 0ull; w.zhi[i] = 0; }
    for (int i = lane; i < nS; i += 32) Kacc[i] = 0u;
    __syncwarp();
    const uint32_t iter = p.state->iter;
    const long bs = (long)gridDim.x * THREADS;
    double *beta = V.beta + (size_t)blockIdx.x * THREADS + tid;
    const unsigned long long chunks = V.coff[G], work = (unsigned long long)p.chains * chunks;
    unsigned long long c_paths = 0; int err = 0;
    UnifCount ctx; ctx.p = &p; ctx.Nacc = w.Nacc; ctx.n = n; ctx.out_idx = 0;
    for (;;) {
        unsigned long long f = 0;
        if (lane == 0) f = atomicAdd(V.next, 1ull);
        f = __shfl_sync(FULL, f, 0);
        if (f >= work) break;
        const unsigned c = (unsigned)(f / chunks);
        const unsigned long long r = f - (unsigned long long)c * chunks;
        int g = 0;
        while (V.coff[g + 1] <= r) g++;
        const unsigned long long j0 = V.gofs[g] + (r - V.coff[g]) * 32ull, j = j0 + (unsigned long long)lane;
        const int unit = (int)c * G + g;
        const double *utab = tab + (size_t)unit * tabd, *model = p.model + (size_t)unit * ML.total;
        if (j < V.gofs[g + 1]) {
            const uint32_t ol = V.perm[j];
            pht_stream st; st.k0 = p.ckeys[2 * c]; st.k1 = p.ckeys[2 * c + 1];
            pht_stream_seek(&st, iter, p.obs_rank + ol * p.obs_world, 0u, 0u);
            ctx.out_idx = (long)ol - p.first;
            const unsigned long long v0 = V.voff[j];
            const int m = (int)(V.voff[j + 1] - v0);
            int B = 0;
            const int e = pht_unif_emis_path(utab, n, cap, model + ML.s, model + ML.scale, model + ML.cum, model + ML.pi, V.y[j], V.cens[j],
                                             V.u ? V.u[j] : INFINITY, m, V.vt + v0, V.vm + v0, X.E + (size_t)c * nS, S, beta, bs, &st,
                                             Za + tid, Zb + tid, THREADS, &ctx, &B);
            err |= e;
            path_flush<THREADS>(p, n, Za, w.zlo, w.zhi, w.Bacc, B, ctx.out_idx);
            if (e == 0 && p.outB == nullptr)
                for (int q = 1; q <= m; q++) atomicAdd(&Kacc[(int)beta[(long)q * n * bs] * S + (int)V.vm[v0 + q - 1]], 1u);
            c_paths++;
        }
        __syncwarp();
        if (p.outB == nullptr) {
            unsigned long long *gs = reinterpret_cast<unsigned long long *>(p.stats + (size_t)unit * stats_len(n));
            for (int i = lane; i < n * n; i += 32) if (w.Nacc[i]) { atomicAdd(&gs[i], (unsigned long long)w.Nacc[i]); w.Nacc[i] = 0u; }
            for (int i = lane; i < n; i += 32) {
                if (w.Bacc[i]) { atomicAdd(&gs[n * n + i], (unsigned long long)w.Bacc[i]); w.Bacc[i] = 0u; }
                if (w.zlo[i]) { atomicAdd(&gs[n * n + n + i], w.zlo[i]); w.zlo[i] = 0ull; }
                if (w.zhi[i]) { atomicAdd(&gs[n * n + 2 * n + i], (unsigned long long)w.zhi[i]); w.zhi[i] = 0; }
            }
            unsigned long long *Kc = X.K + (size_t)c * nS;
            for (int i = lane; i < nS; i += 32) if (Kacc[i]) { atomicAdd(&Kc[i], (unsigned long long)Kacc[i]); Kacc[i] = 0u; }
        }
        __syncwarp();
    }
    if (err) atomicOr(&p.state->error, err);
    for (int o = 16; o > 0; o >>= 1) c_paths += __shfl_down_sync(FULL, c_paths, o);
    if (lane == 0) atomicAdd(&p.state->counters[PHT_CNT_PATHS], c_paths);
}

int pht_unif_emis_grid_blocks(int device, int n, int S) {
    const size_t smem = unif_emis_smem<PHT_UNIF_PANEL_THREADS>(n, S);
    int per_sm = 0, sms = 0;
    if (cudaFuncSetAttribute(k_unif_emis_paths<PHT_UNIF_PANEL_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_unif_emis_paths<PHT_UNIF_PANEL_THREADS>, PHT_UNIF_PANEL_THREADS, smem) != cudaSuccess) return -1;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return -1;
    return per_sm * sms;
}

cudaError_t pht_launch_unif_emis(const SweepParams &p, const double *tab, const UnifPanel &V, const UnifEmis &X, int grid_blocks, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(V.next, 0, sizeof(unsigned long long), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(X.K, 0, sizeof(unsigned long long) * (size_t)p.chains * p.n * X.S, st);
    if (e != cudaSuccess) return e;
    k_unif_emis_paths<PHT_UNIF_PANEL_THREADS><<<grid_blocks, PHT_UNIF_PANEL_THREADS, unif_emis_smem<PHT_UNIF_PANEL_THREADS>(p.n, X.S), st>>>(p, tab, V, X);
    return cudaGetLastError();
}

/* block c: chain c's E rows.  k_update has advanced the sweep, so this sweep is iter - 1 and its row res_row - 1.  Cell
 * (c, o) with alpha > 0 draws Gamma(alpha + K, 1) on parameter sub-stream m + n + c S + o; each row is normalised in index
 * order, as pi is; cells with alpha = 0 stay 0. */
__global__ void __launch_bounds__(128) k_emis_update(UpdateParams p, UnifEmis X) {
    __shared__ double gam[PHT_NMAX * PHT_MAX_STAGES];
    const int n = p.n, S = X.S, nS = n * S, c = blockIdx.x;
    const uint32_t iter = p.state->iter - 1u, row = p.state->res_row - 1u;
    const uint32_t k0 = p.ckeys ? p.ckeys[2 * c] : p.k0, k1 = p.ckeys ? p.ckeys[2 * c + 1] : p.k1;
    double *E = X.E + (size_t)c * nS;
    const unsigned long long *K = X.K + (size_t)c * nS;
    for (int i = threadIdx.x; i < nS; i += blockDim.x) {
        double v = 0.0;
        if (X.alpha[i] > 0.0) {
            pht_stream st; st.k0 = k0; st.k1 = k1;
            pht_stream_seek(&st, iter, PHT_OBS_PARAM, (uint32_t)(p.m + n + i), 0);
            v = pht_rgamma(&st, X.alpha[i] + (double)K[i], 1.0);
        }
        gam[i] = v;
    }
    __syncthreads();
    for (int r = threadIdx.x; r < n; r += blockDim.x) {
        double sum = 0.0;
        for (int o = 0; o < S; o++) sum += gam[r * S + o];
        for (int o = 0; o < S; o++) {
            const double v = X.alpha[r * S + o] > 0.0 ? gam[r * S + o] / sum : 0.0;
            E[r * S + o] = v;
            if (X.Eres != nullptr && row < (uint32_t)p.res_rows) X.Eres[((size_t)c * p.res_rows + row) * nS + r * S + o] = v;
        }
    }
}

cudaError_t pht_launch_emis_update(const UpdateParams &u, const UnifEmis &X, cudaStream_t st) {
    k_emis_update<<<u.chains, 128, 0, st>>>(u, X);
    return cudaGetLastError();
}

size_t pht_unif_entry_scan_bytes(long count) {
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveScan(nullptr, bytes, (const unsigned *)nullptr, (unsigned long long *)nullptr, cuda::std::plus<>(),
                                   0ull, count + 1);
    return bytes;
}

int pht_unif_ghost_grid_blocks(int device, int n) {
    const size_t smem = UnifSmem<UNIF_THREADS>::bytes(n);
    int per_sm = 0, sms = 0;
    if (cudaFuncSetAttribute(k_unif_ghosts<UNIF_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_unif_ghosts<UNIF_THREADS>, UNIF_THREADS, smem) != cudaSuccess) return -1;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return -1;
    return per_sm * sms;
}

cudaError_t pht_launch_unif_entry(const UpdateParams &u, const SweepParams &p, const double *tab, const UnifEntry &E, int ghost_blocks,
                                  int stages, cudaStream_t st) {
    if (stages & PHT_ENTRY_COUNTS) {
        k_unif_entry_table<<<1, UNIF_TABLE_THREADS, 0, st>>>(u, tab, E.etab);
        long blocks = (E.count + 1 + 255) / 256;
        if (blocks > E.count_blocks) blocks = E.count_blocks;
        k_unif_entry_count<<<(unsigned)blocks, 256, 0, st>>>(p, tab, E.etab, E.a, E.obs, E.first, E.count, E.M);
        size_t bytes = E.scan_bytes;
        const cudaError_t e = cub::DeviceScan::ExclusiveScan(E.scan_tmp, bytes, (const unsigned *)E.M, E.off, cuda::std::plus<>(),
                                                             0ull, E.count + 1, st);
        if (e != cudaSuccess) return e;
    }
    if (stages & PHT_ENTRY_GHOSTS) {
        const cudaError_t e = cudaMemsetAsync(E.next, 0, sizeof(unsigned long long), st);
        if (e != cudaSuccess) return e;
        k_unif_ghosts<UNIF_THREADS><<<ghost_blocks, UNIF_THREADS, UnifSmem<UNIF_THREADS>::bytes(p.n), st>>>(
            p, tab, E.a, E.obs, E.first, E.count, E.off, E.next);
    }
    return cudaGetLastError();
}

cudaError_t pht_unif_init(double *tab, int n, int cap, int chains, cudaStream_t st) {
    k_unif_lgk<<<chains, 32, 0, st>>>(tab, n, cap);
    return cudaGetLastError();
}

size_t pht_unif_table_doubles(int n, int cap) { return (size_t)pht_unif_layout_make(n, cap).total; }

cudaError_t pht_launch_unif_table(const UpdateParams &p, double *tab, double tmax, cudaStream_t st) {
    const size_t smem = sizeof(double) * (size_t)(3 * p.n * p.n + 7 * p.n);
    k_unif_table<<<p.chains * p.groups, UNIF_TABLE_THREADS, smem, st>>>(p, tab, tmax);
    return cudaGetLastError();
}

int pht_unif_grid_blocks(int device, int n, bool chains) {     /* chains: the walker (several chains or groups) */
    const size_t smem = UnifSmem<UNIF_THREADS>::bytes(n);
    int per_sm = 0, sms = 0;
    const void *k = chains ? (const void *)k_unif_chain_paths<UNIF_THREADS> : (const void *)k_unif_paths<UNIF_THREADS>;
    if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, UNIF_THREADS, smem) != cudaSuccess) return -1;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return -1;
    return per_sm * sms;
}

cudaError_t pht_launch_unif(const SweepParams &p, const double *tab, const unsigned long long *gofs, int grid_blocks, cudaStream_t st) {
    if ((p.chains > 1 || p.groups > 1) && p.outB == nullptr)
        k_unif_chain_paths<UNIF_THREADS><<<grid_blocks, UNIF_THREADS, UnifSmem<UNIF_THREADS>::bytes(p.n), st>>>(p, tab, gofs);
    else k_unif_paths<UNIF_THREADS><<<grid_blocks, UNIF_THREADS, UnifSmem<UNIF_THREADS>::bytes(p.n), st>>>(p, tab);
    return cudaGetLastError();
}
