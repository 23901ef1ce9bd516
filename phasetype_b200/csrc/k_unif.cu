/*
 * k_unif.cu -- the uniformisation path sampler (method 64) for sm_100a: exact conditional paths for any
 * sub-generator (Hobolth & Stone 2009, section 3.3), for exact, right-, interval- and left-censored observations.
 * Law, table, truncation and draw order: pht_unif.h, which this file and the host restatement share.
 *
 *   k_unif_lgk     once per engine: log k! for k < capacity
 *   k_unif_table   once per sweep (in place of k_spectral_solve): lambda, R = I + S/lambda, r = s/lambda and the
 *                  powers R^k, pi R^k, g_k for k <= K_sweep = K(lambda t_max), by sequential products.  One block: the
 *                  products are a chain of K_sweep dependent steps, each n^2 + 2n dot products of length n, so one
 *                  step is one pass of the block over the entries with the previous power in shared memory.
 *   k_unif_paths   one observation per lane, persistent warps refilled from the global counter (Dispenser); the two
 *                  per-lane n-vectors of scratch live in shared-memory slabs (stride THREADS), the powers in global
 *                  memory (33 MB at n = 32 and full capacity; what a sweep touches stays in L2).
 *
 * Bound: FP64 issue.  Per observation the sampler evaluates ~3 K(lambda y) Poisson weights (one pht_exp each) and
 * ~K(lambda y) n multiply-adds for the end-state weights, plus n per uniformised event; the observations are handed out
 * by decreasing y (k_sort.cu), so the lanes of a warp run similar K.
 */
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

__global__ void k_unif_lgk(double *tab, int n, int cap) {
    if (threadIdx.x == 0 && blockIdx.x == 0) pht_unif_lgk_fill(tab + pht_unif_layout_make(n, cap).lgk, cap);
}

__global__ void __launch_bounds__(UNIF_TABLE_THREADS) k_unif_table(UpdateParams p, double *tab, double tmax) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = p.n, nn = n * n, tid = threadIdx.x, cap = PHT_UNIF_CAP;
    const ModelLayout ML = ModelLayout::make(n, p.m);
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    const double *S = p.model + ML.S, *s = p.model + ML.s, *pi = p.model + ML.pi;
    double *sR = reinterpret_cast<double *>(smem_raw), *sr = sR + nn;
    double *P0 = sr + n, *P1 = P0 + nn, *q0 = P1 + nn, *q1 = q0 + n, *g0 = q1 + n, *g1 = g0 + n;
    const double lam = pht_unif_lambda(n, S);
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

cudaError_t pht_unif_init(double *tab, int n, int cap, cudaStream_t st) {
    k_unif_lgk<<<1, 32, 0, st>>>(tab, n, cap);
    return cudaGetLastError();
}

size_t pht_unif_table_doubles(int n, int cap) { return (size_t)pht_unif_layout_make(n, cap).total; }

cudaError_t pht_launch_unif_table(const UpdateParams &p, double *tab, double tmax, cudaStream_t st) {
    const size_t smem = sizeof(double) * (size_t)(3 * p.n * p.n + 7 * p.n);
    k_unif_table<<<1, UNIF_TABLE_THREADS, smem, st>>>(p, tab, tmax);
    return cudaGetLastError();
}

int pht_unif_grid_blocks(int device, int n) {
    const size_t smem = UnifSmem<UNIF_THREADS>::bytes(n);
    int per_sm = 0, sms = 0;
    if (cudaFuncSetAttribute(k_unif_paths<UNIF_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_unif_paths<UNIF_THREADS>, UNIF_THREADS, smem) != cudaSuccess) return -1;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return -1;
    return per_sm * sms;
}

cudaError_t pht_launch_unif(const SweepParams &p, const double *tab, int grid_blocks, cudaStream_t st) {
    k_unif_paths<UNIF_THREADS><<<grid_blocks, UNIF_THREADS, UnifSmem<UNIF_THREADS>::bytes(p.n), st>>>(p, tab);
    return cudaGetLastError();
}
