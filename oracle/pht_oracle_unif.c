/*
 * pht_oracle_unif.c -- CPU restatement of the uniformisation path sampler (method 64; TEST INFRASTRUCTURE ONLY, like
 * pht_oracle.c).  The per-observation law, draw order and arithmetic are those of phasetype_b200/csrc/pht_unif.h, built
 * here for the host (as pht_eigen.h is): table of R^k, pi R^k and g_k by sequential products, one path per observation
 * on Philox sub-stream 0 of (sweep, global observation).  It includes pht_oracle.c for the Philox streams, the
 * generator assembly, the embedded chain and the start distribution, and sums the statistics into the same fixed point.
 * Built by pyoracle_unif.build() into _build/libphtoracle_unif.so, a library of its own.
 *
 *   int pho_unif_table(n, S, s, pi, tmax, cap, tab)        -> K_sweep, or -1 when it does not fit the table
 *   int pho_unif_paths(seed, iter, obs0, stride, count, y, cens, u, pi, n, S, s, cap, outB, outN, outz)
 *   int pho_unif_sweep_stats(seed, iter, first, n, m, T, C, theta, y, l, cens, u, pi, rank, world, zbits, cap,
 *                            Nacc, Bacc, zfix)
 * u may be NULL (no bounds), pi may be NULL (e1).  The return value of the last two is 0 or the error bit the engine
 * would raise (256: table too small, 512: a draw with only zero weights).
 */
#include "pht_oracle.c"

typedef struct { int *N; int n; } pho_unif_ctx;
#define PHT_UNIF_CTX pho_unif_ctx
#define PHT_UNIF_COUNT(ctx, from, to) ((ctx)->N[(from) + (to) * (ctx)->n]++)
#include "../phasetype_b200/csrc/pht_unif.h"

int pho_unif_table(int n, const double *S, const double *s, const double *pi, double tmax, int cap, double *tab) {
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    pht_unif_lgk_fill(tab + L.lgk, cap);
    const double lam = pht_unif_lambda(n, S);
    double *R = tab + L.R, *r = tab + L.r;
    for (int j = 0; j < n; j++) for (int i = 0; i < n; i++) R[i + j * n] = pht_unif_R_entry(n, S, lam, i, j);
    for (int i = 0; i < n; i++) r[i] = s[i] / lam;
    int K = pht_unif_K(lam * tmax), rc = K;
    if (K >= cap) { K = cap - 1; rc = -1; }
    int npos = 0, a1 = 0;
    for (int i = n - 1; i >= 0; i--) if (pi[i] > 0.0) { npos++; a1 = i; }
    tab[0] = lam; tab[1] = K; tab[2] = npos; tab[3] = a1;
    double *P = tab + L.P, *q = tab + L.q, *g = tab + L.g;
    for (int e = 0; e < n * n; e++) P[e] = (e % n == e / n) ? 1.0 : 0.0;
    for (int i = 0; i < n; i++) { q[i] = pi[i]; g[i] = 0.0; }
    for (int k = 0; k < K; k++) {
        const double *Pk = P + k * n * n, *qk = q + k * n, *gk = g + k * n;
        double *Pn = P + (k + 1) * n * n, *qn = q + (k + 1) * n, *gn = g + (k + 1) * n;
        for (int j = 0; j < n; j++) for (int i = 0; i < n; i++) Pn[i + j * n] = pht_unif_P_entry(n, Pk, R, i, j);
        for (int j = 0; j < n; j++) qn[j] = pht_unif_q_entry(n, qk, R, j);
        for (int i = 0; i < n; i++) gn[i] = pht_unif_g_entry(n, gk, R, r, i);
    }
    return rc;
}

/* the model pieces the sampler reads besides the table, computed as k_assemble does */
static void unif_model(int n, const double *S, const double *s, double *scale, double *cum) {
    double *P = (double *)calloc((size_t)n * n, sizeof(double)), *Pfull = (double *)calloc((size_t)n * (n + 1), sizeof(double));
    pho_embedded(n, S, s, P, Pfull);
    for (int i = 0; i < n; i++) {
        scale[i] = 1.0 / -S[i + i * n];
        double sofar = 0.0;
        for (int k = 0; k <= n; k++) { sofar += Pfull[i + k * n]; cum[i * (n + 1) + k] = sofar; }
    }
    free(P); free(Pfull);
}

int pho_unif_paths(uint64_t seed, uint32_t iter, long obs0, long stride, long count, const double *y, const int *cens,
                   const double *u, const double *pi_in, int n, const double *S, const double *s, int cap,
                   int *outB, int *outN, double *outz) {
    double *pi = (double *)calloc(n, sizeof(double));
    if (pi_in) for (int i = 0; i < n; i++) pi[i] = pi_in[i];
    else pi[0] = 1.0;
    double tmax = 0.0;
    for (long k = 0; k < count; k++) {
        if (y[k] > tmax) tmax = y[k];
        if (u && cens[k] && u[k] <= 1.7976931348623157e308 && u[k] - y[k] > tmax) tmax = u[k] - y[k];
    }
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    double *tab = (double *)calloc((size_t)L.total, sizeof(double));
    double *scale = (double *)calloc(n, sizeof(double)), *cum = (double *)calloc((size_t)(n + 1) * (n + 1), sizeof(double));
    double *zb = (double *)calloc(n, sizeof(double));
    int rc = 0;
    pho_unif_table(n, S, s, pi, tmax, cap, tab);
    unif_model(n, S, s, scale, cum);
    for (long k = 0; k < count; k++) {
        pht_stream st = stream_for(seed, iter, (uint32_t)(obs0 + k * stride));
        int *N = outN + (size_t)k * n * n;
        memset(N, 0, sizeof(int) * (size_t)n * n);
        pho_unif_ctx ctx; ctx.N = N; ctx.n = n;
        rc |= pht_unif_path(tab, n, cap, s, scale, cum, pi, y[k], cens[k], u ? u[k] : INFINITY, &st,
                            outz + (size_t)k * n, zb, 1, &ctx, &outB[k]);
    }
    free(pi); free(tab); free(scale); free(cum); free(zb);
    return rc;
}

int pho_unif_sweep_stats(uint64_t seed, uint32_t iter, int first, int n, int m, const int *T, const double *C,
                         const double *theta, const double *y, long l, const int *censored, const double *u, const double *pi,
                         int rank, int world, int zbits, int cap, long long *Nacc, long long *Bacc, long long *zfix) {
    (void)m;
    const int n1 = n + 1;
    long cnt = 0;
    for (long i = rank; i < l; i += world) cnt++;
    double *TT = (double *)calloc((size_t)n1 * n1, sizeof(double)), *S = (double *)calloc((size_t)n * n, sizeof(double));
    double *s = (double *)calloc(n, sizeof(double));
    double *yl = (double *)malloc(sizeof(double) * (size_t)(cnt + 1)), *ul = (double *)malloc(sizeof(double) * (size_t)(cnt + 1));
    int *cl = (int *)malloc(sizeof(int) * (size_t)(cnt + 1));
    int *B = (int *)malloc(sizeof(int) * (size_t)(cnt + 1)), *N = (int *)malloc(sizeof(int) * (size_t)(cnt + 1) * n * n);
    double *z = (double *)malloc(sizeof(double) * (size_t)(cnt + 1) * n);
    long k = 0;
    for (long i = rank; i < l; i += world, k++) { yl[k] = y[i]; cl[k] = censored[i]; ul[k] = u ? u[i] : INFINITY; }
    assemble(n, T, C, theta, first, TT, S, s);
    const int rc = pho_unif_paths(seed, iter, rank, world, cnt, yl, cl, ul, pi, n, S, s, cap, B, N, z);
    const double zs = ldexp(1.0, zbits);
    memset(Nacc, 0, sizeof(long long) * (size_t)n * n); memset(Bacc, 0, sizeof(long long) * n); memset(zfix, 0, sizeof(long long) * n);
    for (k = 0; k < cnt; k++) {
        Bacc[B[k]]++;
        for (int c = 0; c < n * n; c++) Nacc[c] += N[(size_t)k * n * n + c];
        for (int i = 0; i < n; i++) { const double v = z[(size_t)k * n + i]; if (v != 0.0) zfix[i] += llrint(v * zs); }
    }
    free(TT); free(S); free(s); free(yl); free(ul); free(cl); free(B); free(N); free(z);
    return rc;
}
