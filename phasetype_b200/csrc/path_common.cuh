/*
 * path_common.cuh -- pieces shared by the per-observation path kernels (k_dcs.cu, k_ecs.cu):
 * warp-level observation dispenser, per-path uniform stream, per-lane shared-memory slabs and
 * the reduction of a finished path into the sweep statistics.
 */
#ifndef PHT_PATH_COMMON_CUH
#define PHT_PATH_COMMON_CUH

#include "engine_internal.h"
#include "pht_philox.h"

#define PATH_CHUNK 32u          /* observations a warp takes from the global counter at once */

/* warp-uniform dispenser of observation indices [obs_begin, obs_end) */
struct Dispenser {
    unsigned long long next, end, obs_begin, obs_end;
    bool exhausted;
    __device__ __forceinline__ void init(const SweepParams &p) {
        const bool per_obs = p.outB != nullptr;
        obs_begin = per_obs ? (unsigned long long)p.first : 0ull;
        obs_end = per_obs ? (unsigned long long)(p.first + p.count) : (unsigned long long)p.l_local;
        next = end = 0ull; exhausted = false;
    }
    /* every lane of the warp calls this with the same `idle` ballot; returns the observation index for this
     * lane or ~0ull when it got none */
    __device__ __forceinline__ unsigned long long take(const SweepParams &p, unsigned idle, bool me_idle) {
        return take_from(&p.state->next_obs, idle, me_idle);
    }
    /* the same from another counter (method 64 with several chains: one counter per chain) */
    __device__ __forceinline__ unsigned long long take_from(unsigned long long *counter, unsigned idle, bool me_idle) {
        const unsigned FULL = 0xffffffffu; const int lane = threadIdx.x & 31;
        if (next == end && !exhausted) {
            unsigned long long base = 0;
            if (lane == 0) base = obs_begin + atomicAdd(counter, (unsigned long long)PATH_CHUNK);
            base = __shfl_sync(FULL, base, 0);
            next = base < obs_end ? base : obs_end;
            end = base + PATH_CHUNK < obs_end ? base + PATH_CHUNK : obs_end;
            if (next == end) exhausted = true;
        }
        const unsigned avail = (unsigned)(end - next);
        const unsigned rank = __popc(idle & ((1u << lane) - 1u));
        const unsigned long long mine = (me_idle && rank < avail) ? next + rank : ~0ull;
        const unsigned cnt = __popc(idle);
        next += cnt < avail ? cnt : avail;
        return mine;
    }
};

/* One out-of-line copy of the Philox block function: the path kernels draw uniforms at many places of a large,
 * divergent loop body, and inlining ~70 instructions at each of them costs instruction-cache misses (the DCS loop
 * stalled on `no_instruction` more than on anything else: profiles/r1c_dcs_ncu_full.md). */
static __device__ __noinline__ pht_u32x4 pht_philox_call(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
    return pht_philox4x32_10(c0, c1, c2, c3, k0, k1);
}

/* sequential uniforms of one path: sub-stream `sub` of (iter, observation); the live ECS / DCS samplers draw a whole
 * path from sub-stream 0, the MH variants (MhChain below) give every chain of an observation its own sub-stream */
struct PathRng {
    uint32_t obs, b, sub; double spare; bool odd;
    __device__ __forceinline__ void seek(uint32_t obs_global) { obs = obs_global; b = 0; sub = 0u; odd = false; spare = 0.0; }
    __device__ __forceinline__ double next(const SweepParams &p, uint32_t iter) {
        if (odd) { odd = false; return spare; }
        pht_u32x4 r = pht_philox_call(b++, sub, obs, iter, p.k0, p.k1);
        spare = pht_u01(r.v[2], r.v[3]); odd = true;
        return pht_u01(r.v[0], r.v[1]);
    }
    /* position on draw 0 (skip_first: draw 1) of sub-stream s of the same observation */
    __device__ __forceinline__ void seek_sub(uint32_t s, bool skip_first, const SweepParams &p, uint32_t iter) {
        sub = s; b = 0; odd = false; spare = 0.0;
        if (skip_first) (void)next(p, iter);
    }
};

/* The independence Metropolis-Hastings wrapper of the two sampler variants the reference compiles but never
 * dispatches (src/Simulate_AbsCTMC_gt_Hobolth_DCS.c:268-355, src/Simulate_AbsCTMC_eq_Aslett_DCS.c:49-143), as a
 * per-lane state machine around a chain sampler.  Every chain ends with LJMA_GUI(), the sub-stream hook of the Philox
 * contract, so chain k of an observation IS its sub-stream k and the accept uniform that follows a proposal is draw 0
 * of the next sub-stream (the MHRS layout).  A chain is therefore a pure function of (observation, k, starts at draw
 * 0 or 1), and the wrapper works like the MHRS search / replay split instead of the reference's double buffers: the
 * chains are first run with recording OFF, only (k, offset, last state) of the current one is kept through the accept
 * tests, and the chain that wins is run once more with recording ON. */
struct MhChain {
    uint32_t chain, c_chain, kprop; int c_pre;
    bool off, c_off, have_cur, rec, cens;
    __device__ __forceinline__ void begin(bool censored) {
        chain = 0u; c_chain = 0u; kprop = 0u; c_pre = 0; off = false; c_off = false; have_cur = false; rec = false; cens = censored;
    }
    /* the chain just simulated ended in state `pre`.  Returns true when it was the recorded replay (the caller adds
     * the path to the statistics and takes the next observation); otherwise (chain, off, rec) describe the chain to
     * run next.  RETRY_PROPOSALS: an invalid proposal (s[pre] == 0) is redrawn (eq_Aslett_DCS.c:104-106); the Hobolth
     * variant tests the CURRENT chain there (gt_Hobolth_DCS.c:312), so it never redraws a proposal. */
    template <bool RETRY_PROPOSALS>
    __device__ __forceinline__ bool chain_end(int pre, const double *s, int mhit, const SweepParams &p, uint32_t iter, uint32_t obs) {
        if (rec) return true;
        bool replay = false;
        if (!have_cur) {
            if (s[pre] == 0.0) { chain++; off = false; }                    /* redraw the current chain */
            else {
                have_cur = true; c_chain = chain; c_off = off; c_pre = pre;
                if (cens || mhit == 0) replay = true;                        /* no MH step for a censored observation */
                else { chain++; off = false; }                              /* first proposal */
            }
        } else if (RETRY_PROPOSALS && s[pre] == 0.0) { chain++; off = false; }
        else {
            const pht_u32x4 r = pht_philox_call(0u, chain + 1u, obs, iter, p.k0, p.k1);
            const double U = pht_u01(r.v[0], r.v[1]);
            if (U < s[pre] / s[c_pre]) { c_chain = chain; c_off = off; c_pre = pre; }
            kprop++;
            if ((int)kprop >= mhit) replay = true;
            else { chain++; off = true; }                                    /* the next proposal starts behind the accept uniform */
        }
        if (replay) { rec = true; chain = c_chain; off = c_off; }
        return false;
    }
};

/* reference scan `while (sofar < target) sofar += p[k++]; k--` over a per-lane slab, bounded at n-1 */
template <int THREADS>
__device__ __forceinline__ int slab_scan(const double *slab, int n, double target) {
    double sofar = 0.0; int k = 0;
#pragma unroll 1
    while (sofar < target && k <= n - 1) { sofar += slab[k * THREADS + threadIdx.x]; k++; }
    k--;
    return k < 0 ? 0 : k;
}

/* add one finished path to the statistics (production) or write it out (parity mode) */
template <int THREADS>
__device__ __forceinline__ void path_flush(const SweepParams &p, int n, const double *zslab, unsigned long long *zlo, long long *zhi,
                                           unsigned int *Bacc, int B, long out_idx) {
    const int tid = threadIdx.x;
    if (p.outB != nullptr) {
        p.outB[out_idx] = B;
#pragma unroll 1
        for (int i = 0; i < n; i++) p.outz[out_idx * n + i] = zslab[i * THREADS + tid];
    } else {
        atomicAdd(&Bacc[B], 1u);
        const double zs = pht_u2d((uint64_t)(1023 + p.zbits) << 52);
#pragma unroll 1
        for (int i = 0; i < n; i++) {
            const double v = zslab[i * THREADS + tid];
            if (v != 0.0) {
                if (!(v * zs < 4.0e18) || !(v * zs > -4.0e18)) atomicOr(&p.state->error, 2);
                pht_zfix_add(zlo, zhi, i, __double2ll_rn(v * zs));
            }
        }
    }
}

__device__ __forceinline__ void count_transition(const SweepParams &p, int n, unsigned int *Nacc, long out_idx, int from, int to) {
    if (p.outN != nullptr) p.outN[(size_t)out_idx * n * n + from + to * n]++;
    else atomicAdd(&Nacc[from + to * n], 1u);
}

/* block accumulators -> a statistics block */
template <int THREADS>
__device__ __forceinline__ void block_flush_to(long long *stats, int n, const unsigned int *Nacc, const unsigned int *Bacc,
                                               const unsigned long long *zlo, const long long *zhi) {
    unsigned long long *g = reinterpret_cast<unsigned long long *>(stats);
    for (int i = threadIdx.x; i < n * n; i += THREADS) if (Nacc[i]) atomicAdd(&g[i], (unsigned long long)Nacc[i]);
    for (int i = threadIdx.x; i < n; i += THREADS) {
        if (Bacc[i]) atomicAdd(&g[n * n + i], (unsigned long long)Bacc[i]);
        if (zlo[i]) atomicAdd(&g[n * n + n + i], zlo[i]);
        if (zhi[i]) atomicAdd(&g[n * n + 2 * n + i], (unsigned long long)zhi[i]);
    }
}

/* block accumulators -> global statistics block */
template <int THREADS>
__device__ __forceinline__ void block_flush(const SweepParams &p, int n, const unsigned int *Nacc, const unsigned int *Bacc,
                                            const unsigned long long *zlo, const long long *zhi) {
    if (p.outB != nullptr) return;
    block_flush_to<THREADS>(p.stats, n, Nacc, Bacc, zlo, zhi);
}

#endif
