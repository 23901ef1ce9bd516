/*
 * pht_oracle_misclass.c -- CPU build of the emission form of the panel sampler (method 64 with stage visits,
 * pht_engine_set_stage_visits; TEST INFRASTRUCTURE ONLY, like pht_oracle.c): pht_unif_emis_path of
 * phasetype_b200/csrc/pht_unif.h, next to the per-observation sampler of pht_oracle_unif.c, which it includes (table, model
 * pieces, streams).  tests/test_misclass_oracle.py checks its law against exact values; tests/test_misclass_gpu.py checks
 * the engine against it bit for bit.  Built by pyoracle_misclass.build() into _build/libphtoracle_misclass.so.
 *
 *   int pho_misclass_paths(seed, iter, count, obs, y, cens, u, pi, voff, vt, vstage, E, S, n, Sm, s, cap, tmax,
 *                          outB, outN, outz, outX)
 *   int pho_misclass_sweep_stats(seed, iter, first, n, T, C, theta, l, obs, y, cens, u, pi, voff, vt, vstage, E, S, zbits,
 *                                cap, Nacc, Bacc, zfix, K)
 * As pho_panel_paths / pho_panel_sweep_stats of pht_oracle_panel.c with stage indices vstage read through E (n x S,
 * row-major) in place of masks; outX (may be NULL) receives the drawn visit states, K (n x S) the visits by (drawn phase,
 * stage read).  The return value is 0 or the engine's error bits (256, 512).
 */
#include "pht_oracle_unif.c"

int pho_misclass_paths(uint64_t seed, uint32_t iter, long count, const uint32_t *obs, const double *y, const int *cens,
                       const double *u, const double *pi_in, const int64_t *voff, const double *vt, const uint32_t *vstage,
                       const double *E, int Sn, int n, const double *S, const double *s, int cap, double tmax, int *outB,
                       int *outN, double *outz, int *outX) {
    double *pi = (double *)calloc(n, sizeof(double));
    if (pi_in) for (int i = 0; i < n; i++) pi[i] = pi_in[i];
    else pi[0] = 1.0;
    if (!(tmax > 0.0)) {
        tmax = 0.0;
        for (long k = 0; k < count; k++) {
            if (y[k] > tmax) tmax = y[k];
            if (u && cens[k] && u[k] <= 1.7976931348623157e308 && u[k] - y[k] > tmax) tmax = u[k] - y[k];
        }
    }
    long mmax = 0;
    for (long k = 0; k < count; k++) if (voff[k + 1] - voff[k] > mmax) mmax = (long)(voff[k + 1] - voff[k]);
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    double *tab = (double *)calloc((size_t)L.total, sizeof(double));
    double *scale = (double *)calloc(n, sizeof(double)), *cum = (double *)calloc((size_t)(n + 1) * (n + 1), sizeof(double));
    double *zb = (double *)calloc(n, sizeof(double)), *beta = (double *)calloc((size_t)(mmax + 1) * n, sizeof(double));
    int rc = 0;
    pho_unif_table(n, S, s, pi, tmax, cap, tab);
    unif_model(n, S, s, scale, cum);
    for (long k = 0; k < count; k++) {
        pht_stream st = stream_for(seed, iter, obs ? obs[k] : (uint32_t)k);
        int *N = outN + (size_t)k * n * n;
        memset(N, 0, sizeof(int) * (size_t)n * n);
        pho_unif_ctx ctx; ctx.N = N; ctx.n = n;
        const int m = (int)(voff[k + 1] - voff[k]);
        const double uk = u ? u[k] : INFINITY;
        int e;
        if (m == 0) e = pht_unif_path(tab, n, cap, s, scale, cum, pi, y[k], cens[k], uk, &st, outz + (size_t)k * n, zb, 1, &ctx, &outB[k]);
        else e = pht_unif_emis_path(tab, n, cap, s, scale, cum, pi, y[k], cens[k], uk, m, vt + voff[k], vstage + voff[k], E, Sn, beta, 1,
                                    &st, outz + (size_t)k * n, zb, 1, &ctx, &outB[k]);
        rc |= e;
        if (outX) for (int j = 1; j <= m; j++) outX[voff[k] + j - 1] = e ? -1 : (int)beta[(size_t)j * n];
    }
    free(pi); free(tab); free(scale); free(cum); free(zb); free(beta);
    return rc;
}

int pho_misclass_sweep_stats(uint64_t seed, uint32_t iter, int first, int n, const int *T, const double *C, const double *theta,
                             long l, const uint32_t *obs, const double *y, const int *cens, const double *u, const double *pi, const int64_t *voff,
                             const double *vt, const uint32_t *vstage, const double *E, int Sn, int zbits, int cap,
                             long long *Nacc, long long *Bacc, long long *zfix, long long *K) {
    const int n1 = n + 1;
    double *TT = (double *)calloc((size_t)n1 * n1, sizeof(double)), *S = (double *)calloc((size_t)n * n, sizeof(double));
    double *s = (double *)calloc(n, sizeof(double));
    int *B = (int *)malloc(sizeof(int) * (size_t)(l + 1)), *N = (int *)malloc(sizeof(int) * (size_t)(l + 1) * n * n);
    int *X = (int *)malloc(sizeof(int) * (size_t)(voff[l] + 1));
    double *z = (double *)malloc(sizeof(double) * (size_t)(l + 1) * n);
    assemble(n, T, C, theta, first, TT, S, s);
    const int rc = pho_misclass_paths(seed, iter, l, obs, y, cens, u, pi, voff, vt, vstage, E, Sn, n, S, s, cap, 0.0, B, N, z, X);
    const double zs = ldexp(1.0, zbits);
    memset(Nacc, 0, sizeof(long long) * (size_t)n * n); memset(Bacc, 0, sizeof(long long) * n); memset(zfix, 0, sizeof(long long) * n);
    memset(K, 0, sizeof(long long) * (size_t)n * Sn);
    for (long k = 0; k < l; k++) {
        Bacc[B[k]]++;
        for (int c = 0; c < n * n; c++) Nacc[c] += N[(size_t)k * n * n + c];
        for (int i = 0; i < n; i++) { const double v = z[(size_t)k * n + i]; if (v != 0.0) zfix[i] += llrint(v * zs); }
    }
    for (int64_t q = 0; q < voff[l]; q++) if (X[q] >= 0) K[(size_t)X[q] * Sn + vstage[q]]++;
    free(TT); free(S); free(s); free(B); free(N); free(X); free(z);
    return rc;
}
