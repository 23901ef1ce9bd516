/*
 * k_model.cu -- the two single-block kernels that bracket every sweep so the
 * whole Gibbs iteration stays on the device (no host round trip):
 *
 *   k_assemble  theta -> TT, S, s (reference src/PHT_MCMC_Aslett.c:209-246 for the
 *               start values, :365-397 afterwards), embedded chain P / Pfull
 *               (:280-297), rexp scales, running-sum tables for the categorical
 *               scans, and zeroing of the statistics block;
 *   k_update    gather Nsum / zsum per parameter (:340-355) and the conjugate
 *               Gamma draw (:365-366) from the Philox parameter stream.
 *
 * With several chains (method 64, pht_engine_set_chains) both run one block per
 * chain, block c on chain c's model, statistics block, key and result rows.  With
 * groups (pht_engine_set_groups) k_assemble runs one block per (chain, group) unit
 * on the group's T and C, and k_update's block c gathers over the groups of chain c.
 *
 * Row i of every matrix is handled by thread i with the reference's own loop
 * order, so each value is bit-identical to the host computation.
 */
#include "engine_internal.h"
#include "pht_philox.h"
#define PHT_EIGEN_WARP 1          /* on the device the solver is run by one warp in lock step (pht_eigen.h) */
#include "pht_eigen.h"

__global__ void __launch_bounds__(64) k_assemble(UpdateParams p) {
    const int n = p.n, n1 = n + 1, tid = threadIdx.x;
    const ModelLayout L = ModelLayout::make(n, p.m);
    const int c = blockIdx.x;                /* unit: chain c / groups, group c % groups (grid = chains x groups) */
    double *M = p.model + (size_t)c * L.total;
    long long *stats = p.stats + (size_t)c * stats_len(n);
    const double *theta = M + L.theta;
    double *TT = M + L.TT, *S = M + L.S, *s = M + L.s;
    const bool first = p.state->first_assembly != 0;
    const size_t gofs = (size_t)(c % p.groups) * n1 * n1;
    const int *T = p.T + gofs; const double *Cm = p.C + gofs;

    for (int i = tid; i < stats_len(n); i += blockDim.x) stats[i] = 0;
    if (tid == 0 && c == 0) {
        p.state->next_obs = 0ull; p.state->unit_counter = 0ull; p.state->replay_next = 0ull;
        p.state->n_items = 0u; p.state->n_pend[0] = 0u; p.state->n_pend[1] = 0u; p.state->n_done = 0u;
    }
    if (tid == 0 && p.cnext != nullptr) p.cnext[c] = 0ull;
    if (tid <= n) {
        const int i = tid;
        for (int j = 0; j <= n; j++) {
            const int v = T[i + j * n1];
            if (j != i || v != 0) TT[i + j * n1] = v ? theta[v - 1] * Cm[i + j * n1] : 0.0;
        }
        /* diagonal = -(row sum): ascending columns when assembled from the start
         * values (:215,229), descending afterwards (TTDiag is a prepend list, :226,389-393) */
        double acc = 0.0;
        if (first) { for (int j = 0; j <= n; j++) if (T[i + j * n1] != 0) acc -= TT[i + j * n1]; }
        else       { for (int j = n; j >= 0; j--) if (T[i + j * n1] != 0) acc -= TT[i + j * n1]; }
        if (i < n || first) TT[i + i * n1] = acc;
    }
    __syncthreads();
    if (tid < n) {
        const int i = tid;
        for (int j = 0; j < n; j++) S[i + j * n] = TT[i + j * n1];
        s[i] = TT[i + n * n1];
        const double Sii = S[i + i * n];
        M[L.scale + i] = 1.0 / -Sii;
        /* embedded chain, src/PHT_MCMC_Aslett.c:280-297 */
        double *P = M + L.P, *Pf = M + L.Pfull;
        double rsumfull = 0.0;
        for (int j = 0; j < n; j++) {
            const double v = -S[i + j * n] / Sii;
            P[i + j * n] = v; Pf[i + j * n] = v;
            rsumfull += v;
        }
        const double rsum = rsumfull - P[i + i * n];
        Pf[i + n * n] = -s[i] / Sii;
        rsumfull += Pf[i + n * n];
        rsumfull -= Pf[i + i * n];
        Pf[i + i * n] = 0.0; P[i + i * n] = 0.0;
        for (int j = 0; j < n; j++) {
            P[i + j * n] = P[i + j * n] / rsum;
            Pf[i + j * n] = Pf[i + j * n] / rsumfull;
        }
        Pf[i + n * n] = Pf[i + n * n] / rsumfull;
        /* running sums in scan order: cum[i][k] = ((p0 + p1) + ...) + pk */
        double *cum = M + L.cum + i * n1;
        double sofar = 0.0;
        for (int k = 0; k <= n; k++) { sofar += Pf[i + k * n]; cum[k] = sofar; }
    }
    if (tid == n) {
        /* running sums of the start distribution (row n of the scan tables).  pi is e1 unless the caller set another
         * one or switched its Dirichlet update on (the reference fixes it to e1: src/PHT_MCMC_Aslett.c:190-193) */
        const double *pi = M + L.pi; double *cum = M + L.cum + n * n1;
        double sofar = 0.0;
        for (int k = 0; k < n; k++) { sofar += pi[k]; cum[k] = sofar; }
        cum[n] = sofar;
    }
}

__global__ void __launch_bounds__(128) k_update(UpdateParams p) {
    const int n = p.n, n1 = n + 1, m = p.m;
    const ModelLayout L = ModelLayout::make(n, m);
    const uint32_t iter = p.state->iter;
    const uint32_t row = p.state->res_row;
    /* chain c (grid = chains): its model and statistics blocks (one per group, c G .. c G + G - 1), key and rows */
    const int c = blockIdx.x, G = p.groups;
    double *model = p.model + (size_t)c * G * L.total;
    const long long *stats = p.stats + (size_t)c * G * stats_len(n);
    const uint32_t k0 = p.ckeys ? p.ckeys[2 * c] : p.k0, k1 = p.ckeys ? p.ckeys[2 * c + 1] : p.k1;
    double *res = p.res ? p.res + (size_t)c * p.res_rows * m : nullptr;
    double *pires = p.pires ? p.pires + (size_t)c * p.res_rows * n : nullptr;
    const double zscale = pht_u2d((uint64_t)(1023 - p.zbits) << 52);      /* 2^-zbits */
    /* some rank raised its error word this sweep: every rank learns it here and stops at the next synchronisation */
    if (threadIdx.x == 0 && stats[stats_len(n) - 1] != 0 && p.state->error == 0) atomicOr(&p.state->error, 128);
    for (int v = threadIdx.x; v < m; v += blockDim.x) {
        long long Nsum = 0; double zsum = 0.0;
        /* groups in ascending order; within a group the reference walks prepend lists, i.e. cells in reverse insertion
         * order (:340-355) */
        for (int g = 0; g < G; g++) {
            const long long *gs = stats + (size_t)g * stats_len(n);
            const long long *Nacc = gs, *zlo = gs + n * n + n, *zhi = gs + n * n + 2 * n;
            const double *Cg = p.C + (size_t)g * n1 * n1;
            for (int c = p.var_ptr[g * m + v + 1] - 1; c >= p.var_ptr[g * m + v]; c--) {
                const int i = p.cell_i[c], j = p.cell_j[c];
                Nsum += (j == n) ? Nacc[i + i * n] : Nacc[i + j * n];
                /* the two limbs of the fixed-point total; it must fit the int64 it is converted from (else: error word 2) */
                const __int128 tot = ((__int128)zhi[i] << 32) + (__int128)(unsigned long long)zlo[i];
                if (tot > (__int128)0x7fffffffffffffffLL || tot < -(__int128)0x7fffffffffffffffLL) atomicOr(&p.state->error, 2);
                const double zi = (double)(long long)tot * zscale;
                zsum += zi / Cg[i + j * n1];
            }
        }
        pht_stream st; st.k0 = k0; st.k1 = k1;
        pht_stream_seek(&st, iter, PHT_OBS_PARAM, (uint32_t)v, 0);
        const double th = pht_rgamma(&st, p.nu[v] + (double)Nsum, 1.0 / (p.zeta[v] + zsum));   /* :366 */
        for (int g = 0; g < G; g++) model[(size_t)g * L.total + L.theta + v] = th;     /* theta lives in every group's block */
        if (res != nullptr && row < (uint32_t)p.res_rows) res[(size_t)row * m + v] = th;
    }
    /* start distribution: pi | paths ~ Dirichlet(beta + B), B = start-state counts of the sweep (the conjugate update the
     * reference leaves as FIX ME, src/PHT_MCMC_Aslett.c:190-193; beta is R/phtMCMC2.R:20-21's prior).  Drawn as n
     * Gamma(beta_i + B_i, 1) variates from parameter sub-streams m .. m+n-1, normalised in index order. */
    __shared__ double gpi[PHT_NMAX];
    if (p.beta != nullptr) {
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            long long Bsum = 0;                 /* start-state counts summed over the groups: one pi per chain */
            for (int g = 0; g < G; g++) Bsum += stats[(size_t)g * stats_len(n) + n * n + i];
            pht_stream st; st.k0 = k0; st.k1 = k1;
            pht_stream_seek(&st, iter, PHT_OBS_PARAM, (uint32_t)(m + i), 0);
            gpi[i] = pht_rgamma(&st, p.beta[i] + (double)Bsum, 1.0);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (p.beta != nullptr) {
            double sum = 0.0;
            for (int i = 0; i < n; i++) sum += gpi[i];
            for (int i = 0; i < n; i++) {
                const double v = gpi[i] / sum;
                for (int g = 0; g < G; g++) model[(size_t)g * L.total + L.pi + i] = v;
                if (pires != nullptr && row < (uint32_t)p.res_rows) pires[(size_t)row * n + i] = v;
            }
        }
        /* Every block read iter and res_row on entry, so the sweep may advance only once all blocks have: the last block
         * to finish (a ticket taken after its reads) advances it and resets the ticket for the next launch. */
        bool last = gridDim.x == 1;
        if (!last) { __threadfence(); last = atomicAdd(&p.state->update_ticket, 1u) == gridDim.x - 1; }
        if (last) { p.state->update_ticket = 0u; p.state->iter = iter + 1; p.state->first_assembly = 0; p.state->res_row = row + 1; }
    }
}

/* Spectral data for ECS / DCS (reference src/utility.c:87-129 via LJMA_eigen, then the GEMVs of
 * src/PHT_MCMC_Aslett.c:328-332).  This variant takes (evals | Q | Q^-1) supplied by the host -- the parity
 * hook pht_engine_set_spectral -- and derives Q^-1 s and Q^-1 1 in reference-BLAS order (dgemv 'N':
 * y_i = sum_j x_j A_ij accumulated over j). */
__global__ void __launch_bounds__(64) k_spectral_inject(UpdateParams p, const double *inject) {
    const int n = p.n, tid = threadIdx.x;
    const ModelLayout L = ModelLayout::make(n, p.m);
    double *M = p.model;
    for (int i = tid; i < n; i += blockDim.x) { M[L.evals + i] = inject[i]; M[L.evals_im + i] = 0.0; }
    for (int i = tid; i < n * n; i += blockDim.x) { M[L.Q + i] = inject[n + i]; M[L.Qinv + i] = inject[n + n * n + i]; }
    __syncthreads();
    if (tid < n) {
        const int i = tid;
        double ys = 0.0, y1 = 0.0;
        for (int j = 0; j < n; j++) {
            const double a = M[L.Qinv + i + j * n];
            ys += (1.0 * M[L.s + j]) * a;
            y1 += (1.0 * 1.0) * a;
        }
        M[L.Qinv_s + i] = ys; M[L.Qinv_1 + i] = y1;
    }
}

/* The engine's own solver (pht_eigen.h: Hessenberg + shifted QR + Gauss-Jordan), one warp working in shared memory,
 * once per sweep.  The block then forms Q^-1 s and Q^-1 1. */
__global__ void __launch_bounds__(64) k_spectral_solve(UpdateParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = p.n, tid = threadIdx.x;
    const ModelLayout L = ModelLayout::make(n, p.m);
    double *M = p.model;
    /* the solver runs in shared memory, by warp 0 in lock step (pht_eigen.h: independent rows / columns dealt out over the
     * lanes, scalar recurrences computed by all of them; bit-identical to the sequential host code): S is staged in, Q, Q^-1
     * and the eigenvalues are written back by the whole block */
    double *w = reinterpret_cast<double *>(smem_raw);
    double *sS = w + 2 * n * n + 3 * n, *sQ = sS + n * n, *sQi = sQ + n * n, *sev = sQi + n * n;
    for (int i = tid; i < n * n; i += blockDim.x) sS[i] = M[L.S + i];
    __syncthreads();
    if (tid < 32) {
        const int st = pht_eigen_real(n, sS, sev, sQ, sQi, w, w + n * n, w + 2 * n * n,
                                      w + 2 * n * n + n, w + 2 * n * n + 2 * n);
        /* complex pairs (st & 2) are not an error: evals_im marks them and the samplers use the real block form */
        if (tid == 0 && (st & 5)) atomicOr(&p.state->error, 32);
    }
    __syncthreads();
    for (int i = tid; i < n * n; i += blockDim.x) { M[L.Q + i] = sQ[i]; M[L.Qinv + i] = sQi[i]; }
    if (tid < n) {
        const int i = tid;
        M[L.evals + i] = sev[i]; M[L.evals_im + i] = w[2 * n * n + 2 * n + i];
        double ys = 0.0, y1 = 0.0;
        for (int j = 0; j < n; j++) {
            const double a = sQi[i + j * n];
            ys += (1.0 * M[L.s + j]) * a;
            y1 += (1.0 * 1.0) * a;
        }
        M[L.Qinv_s + i] = ys; M[L.Qinv_1 + i] = y1;
    }
}

cudaError_t pht_launch_spectral(const UpdateParams &p, const double *inject, cudaStream_t st) {
    if (inject != nullptr) k_spectral_inject<<<1, 64, 0, st>>>(p, inject);
    else k_spectral_solve<<<1, 64, sizeof(double) * (5 * p.n * p.n + 4 * p.n), st>>>(p);
    return cudaGetLastError();
}

cudaError_t pht_launch_assemble(const UpdateParams &p, cudaStream_t st) {
    k_assemble<<<p.chains * p.groups, 64, 0, st>>>(p);
    return cudaGetLastError();
}
cudaError_t pht_launch_update(const UpdateParams &p, cudaStream_t st) {
    k_update<<<p.chains, 128, 0, st>>>(p);
    return cudaGetLastError();
}

/* before the all-reduce of a multi-GPU sweep: the last word of the statistics block says whether this rank's error
 * word is raised, so the sum tells every rank (k_update) */
__global__ void k_pack_error(long long *stats, int len, const DevState *state) {
    if (threadIdx.x == 0) stats[len - 1] = state->error != 0 ? 1 : 0;
}
/* All-reduce (sum, int64) of the statistics block over the GPUs of the run WITHOUT a library call: every rank stores
 * its block into its slot of every rank's exchange window (NVLink peer stores; its own window included), raises its
 * flag there, waits until every rank's flag has arrived in its own window, and sums the slots it now holds locally,
 * in rank order.  ~len * world 8-byte stores per rank and one flag round trip: the payload is n^2+3n+1 words, so this
 * is a latency-sized exchange (a few microseconds over NVSwitch), captured in the sweep graph like any kernel.
 * Slots and flags are double buffered by the parity of the all-reduce count: a rank can be at most one all-reduce
 * ahead of the slowest (it needs everybody's flag to pass), so the buffer it overwrites has been read by all.
 * The last word of the block says whether this rank's error word is raised, so every rank learns it (k_update). */
__device__ __forceinline__ unsigned long long reduce_timer() {
    unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t;
}
__global__ void __launch_bounds__(256) k_allreduce_peer(const __grid_constant__ ReduceParams p) {
    const int tid = threadIdx.x;
    __shared__ unsigned long long s_epoch;
    if (tid == 0) { p.stats[p.len - 1] = p.state->error != 0 ? 1 : 0; s_epoch = p.state->sepoch + 1ull; }
    __syncthreads();
    const unsigned long long epoch = s_epoch; const int par = (int)(epoch & 1ull);
    for (uint32_t r = 0; r < p.world; r++) {
        volatile long long *dst = p.xpeer[r]->sstats[par][p.rank];
        for (int i = tid; i < p.len; i += blockDim.x) dst[i] = p.stats[i];
    }
    __threadfence_system();
    __syncthreads();
    if (tid < (int)p.world && p.state->xdead == 0u) {
        volatile unsigned long long *mine = &p.xpeer[tid]->sflags[par][p.rank];
        *mine = epoch;
        __threadfence_system();
        volatile unsigned long long *theirs = &p.xw->sflags[par][tid];
        const unsigned long long t0 = reduce_timer();
        while (*theirs < epoch) {
            if (reduce_timer() - t0 > 4000000000ull) { p.state->xdead = 1u; atomicOr(&p.state->error, 64); break; }
        }
        __threadfence_system();
    }
    __syncthreads();
    if (p.state->xdead == 0u) {
        for (int i = tid; i < p.len; i += blockDim.x) {
            long long sum = 0;
            for (uint32_t r = 0; r < p.world; r++) sum += const_cast<volatile long long *>(p.xw->sstats[par][r])[i];
            p.stats[i] = sum;
        }
    } else if (tid == 0) p.stats[p.len - 1] = 1;
    if (tid == 0) p.state->sepoch = epoch;
}
cudaError_t pht_launch_peer_allreduce(const ReduceParams &p, cudaStream_t st) {
    k_allreduce_peer<<<1, 256, 0, st>>>(p);
    return cudaGetLastError();
}

cudaError_t pht_launch_pack_error(const UpdateParams &p, cudaStream_t st) {
    k_pack_error<<<1, 32, 0, st>>>(p.stats, stats_len(p.n), p.state);
    return cudaGetLastError();
}
