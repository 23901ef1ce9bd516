/*
 * pht_oracle_iv.c -- CPU restatement of the MHRS sampler for interval-censored observations (TEST INFRASTRUCTURE ONLY,
 * like pht_oracle.c).  The reference has no upper bound; u[k] bounds observation k's absorption time from above
 * (+inf: none), and the rejection retry of mhrs_draw, `while (t < y)` (src/Simulate_AbsCTMC_gt_Bladt_MHRS.c:49),
 * becomes `while (t < y || t > u)`.  With every u = +inf both entry points return exactly what pho_mhrs_paths /
 * pho_sweep_stats (method MHRS) return.
 *
 * The restatement's helpers (Philox streams, categorical scan, rexp, start distribution, generator assembly) are
 * file-static in pht_oracle.c; this file includes it, so the interval sampler runs the very same arithmetic without
 * that file changing.  Built by pyoracle_iv.build() into _build/libphtoracle_iv.so, a library of its own.
 *
 *   int pho_mhrs_paths_iv(seed, iter, obs0, stride, count, y, cens, u, n, S, s, Pfull, mhit, outB, outN, outz, counters)
 *   int pho_sweep_stats_iv(seed, iter, first, mhit, n, m, T, C, theta, y, l, censored, u, rank, world, zbits,
 *                          Nacc, Bacc, zfix, counters)
 */
#include "pht_oracle.c"

/* mhrs_draw with the restated retry: an attempt survives when it is absorbed at y <= t <= u */
static path_ends mhrs_draw_iv(pht_stream *st, double y, int censored, double u, int n, const double *pi, const double *S,
                              const double *Pfull, double *z2, int *N2, unsigned long long *cnt) {
    double t = 0.0, lastt = 0.0; int B2 = 0, j, lastj = 0;
    while (t < y || t > u) {
        t = 0.0;
        memset(N2, 0, sizeof(int) * (size_t)n * n);
        for (int i = 0; i < n; i++) z2[i] = 0.0;
        B2 = cat_scan(pi, 1, n - 1, runif01(st));
        j = B2; lastt = t; lastj = j;
        while ((t < y && j < n) || (censored && j < n)) {
            t = t + rexp_scale(st, 1.0 / -S[j + j * n]);
            j = cat_scan(Pfull + j, n, n, runif01(st));
            if (cnt) cnt[PHO_C_JUMPS]++;
            if ((t < y && j < n) || (censored && j < n)) {
                z2[lastj] += t - lastt;
                N2[lastj + j * n]++;
                lastj = j; lastt = t;
            }
        }
        next_substream(st);
        if (cnt) cnt[PHO_C_ATTEMPTS]++;
    }
    if (!censored) z2[lastj] += y - lastt; else z2[lastj] += t - lastt;
    N2[lastj + lastj * n]++;
    path_ends e; e.B = B2; e.pre = lastj;
    return e;
}

static path_ends mhrs_observation_iv(pht_stream *st, double y, int censored, double u, int n, const double *pi, const double *S,
                                     const double *s, const double *Pfull, int mhit, double **zc, int **Nc,
                                     double **zp, int **Np, unsigned long long *cnt) {
    path_ends cur = mhrs_draw_iv(st, y, censored, u, n, pi, S, Pfull, *zc, *Nc, cnt);
    while (s[cur.pre] == 0) cur = mhrs_draw_iv(st, y, censored, u, n, pi, S, Pfull, *zc, *Nc, cnt);
    if (!censored) {
        for (int it = 0; it < mhit; it++) {
            path_ends prop = mhrs_draw_iv(st, y, censored, u, n, pi, S, Pfull, *zp, *Np, cnt);
            while (s[prop.pre] == 0) prop = mhrs_draw_iv(st, y, censored, u, n, pi, S, Pfull, *zp, *Np, cnt);
            double U = runif01(st);
            if (U < s[prop.pre] / s[cur.pre]) {
                double *tz = *zc; *zc = *zp; *zp = tz;
                int *tN = *Nc; *Nc = *Np; *Np = tN;
                cur = prop;
            }
        }
    }
    return cur;
}

int pho_mhrs_paths_iv(uint64_t seed, uint32_t iter, long obs0, long stride, long count,
                      const double *y, const int *cens, const double *u, int n, const double *S, const double *s,
                      const double *Pfull, int mhit, int *outB, int *outN, double *outz,
                      unsigned long long *counters) {
    double *pi = (double *)calloc(n, sizeof(double));
    double *za = (double *)calloc(n, sizeof(double)), *zb = (double *)calloc(n, sizeof(double));
    int *Na = (int *)calloc((size_t)n * n, sizeof(int)), *Nb = (int *)calloc((size_t)n * n, sizeof(int));
    if (!pi || !za || !zb || !Na || !Nb) return -1;
    pi_init(pi, n);
    for (long k = 0; k < count; k++) {
        pht_stream st = stream_for(seed, iter, (uint32_t)(obs0 + k * stride));
        double *zc = za, *zp = zb; int *Nc = Na, *Np = Nb;
        path_ends e = mhrs_observation_iv(&st, y[k], cens[k], u[k], n, pi, S, s, Pfull, mhit, &zc, &Nc, &zp, &Np, counters);
        if (counters) counters[PHO_C_PATHS]++;
        outB[k] = e.B;
        memcpy(outN + (size_t)k * n * n, Nc, sizeof(int) * (size_t)n * n);
        memcpy(outz + (size_t)k * n, zc, sizeof(double) * (size_t)n);
    }
    free(pi); free(za); free(zb); free(Na); free(Nb);
    return 0;
}

int pho_sweep_stats_iv(uint64_t seed, uint32_t iter, int first, int mhit, int n, int m, const int *T, const double *C,
                       const double *theta, const double *y, long l, const int *censored, const double *u, int rank, int world,
                       int zbits, long long *Nacc, long long *Bacc, long long *zfix, unsigned long long *counters) {
    (void)m;
    const int n1 = n + 1;
    long cnt = 0;
    for (long i = rank; i < l; i += world) cnt++;
    double *TT = (double *)calloc((size_t)n1 * n1, sizeof(double)), *S = (double *)calloc((size_t)n * n, sizeof(double));
    double *s = (double *)calloc(n, sizeof(double)), *P = (double *)calloc((size_t)n * n, sizeof(double));
    double *Pfull = (double *)calloc((size_t)n * n1, sizeof(double));
    double *yl = (double *)malloc(sizeof(double) * (size_t)(cnt + 1)), *ul = (double *)malloc(sizeof(double) * (size_t)(cnt + 1));
    int *cl = (int *)malloc(sizeof(int) * (size_t)(cnt + 1));
    int *B = (int *)malloc(sizeof(int) * (size_t)(cnt + 1)), *N = (int *)malloc(sizeof(int) * (size_t)(cnt + 1) * n * n);
    double *z = (double *)malloc(sizeof(double) * (size_t)(cnt + 1) * n);
    long k = 0;
    for (long i = rank; i < l; i += world, k++) { yl[k] = y[i]; cl[k] = censored[i]; ul[k] = u[i]; }
    assemble(n, T, C, theta, first, TT, S, s);
    pho_embedded(n, S, s, P, Pfull);
    int rc = pho_mhrs_paths_iv(seed, iter, rank, world, cnt, yl, cl, ul, n, S, s, Pfull, mhit, B, N, z, counters);
    if (rc == 0) {
        const double zs = ldexp(1.0, zbits);
        memset(Nacc, 0, sizeof(long long) * (size_t)n * n); memset(Bacc, 0, sizeof(long long) * n); memset(zfix, 0, sizeof(long long) * n);
        for (k = 0; k < cnt; k++) {
            Bacc[B[k]]++;
            for (int c = 0; c < n * n; c++) Nacc[c] += N[(size_t)k * n * n + c];
            for (int i = 0; i < n; i++) { const double v = z[(size_t)k * n + i]; if (v != 0.0) zfix[i] += llrint(v * zs); }
        }
    }
    free(TT); free(S); free(s); free(P); free(Pfull); free(yl); free(ul); free(cl); free(B); free(N); free(z);
    return rc;
}
