/*
 * pht_oracle_groups.c -- CPU restatement of groups with their own generator structure for the uniformisation sampler
 * (method 64, pht_engine_set_groups; TEST INFRASTRUCTURE ONLY, like pht_oracle.c).  Every observation's path is the
 * existing per-observation sampler (pht_unif.h, via pht_oracle_unif.c) run on its own group's model: the group's S and s
 * assembled from theta with (T_g, C_g), its own table, Philox sub-stream 0 of (sweep, global observation).  The statistics
 * are kept per group, and the update gathers them over the groups in ascending order -- within a group the cells in the
 * reference's prepend-list order, z / C included (pho_update) -- before the one Gamma draw per parameter.  Built by
 * pyoracle_groups.build() into _build/libphtoracle_groups.so, a library of its own.
 *
 *   int pho_groups_sweep_stats(seed, iter, first, n, G, T, C, theta, y, l, cens, u, group, pi, zbits, cap, Nacc, Bacc, zfix)
 *   int pho_groups_update(seed, iter, n, m, G, nu, zeta, T, C, zbits, Nacc, zfix, theta_new)
 * T, C: G structures of (n+1)^2 (column-major); group[k] in 0..G-1; u may be NULL (no bounds), pi NULL (e1).  Nacc, Bacc
 * and zfix receive G blocks (n*n, n, n).  The sweep statistics return 0 or the engine's error bits (256, 512).
 */
#include "pht_oracle_unif.c"

int pho_groups_sweep_stats(uint64_t seed, uint32_t iter, int first, int n, int G, const int *T, const double *C,
                           const double *theta, const double *y, long l, const int *censored, const double *u, const int *group,
                           const double *pi_in, int zbits, int cap, long long *Nacc, long long *Bacc, long long *zfix) {
    const int n1 = n + 1;
    const double zs = ldexp(1.0, zbits);
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    double *pi = (double *)calloc(n, sizeof(double));
    if (pi_in) for (int i = 0; i < n; i++) pi[i] = pi_in[i];
    else pi[0] = 1.0;
    double *TT = (double *)calloc((size_t)n1 * n1, sizeof(double)), *S = (double *)calloc((size_t)n * n, sizeof(double));
    double *s = (double *)calloc(n, sizeof(double)), *scale = (double *)calloc(n, sizeof(double));
    double *cum = (double *)calloc((size_t)n1 * n1, sizeof(double)), *zb = (double *)calloc(n, sizeof(double));
    double *z = (double *)calloc(n, sizeof(double)), *tab = (double *)calloc((size_t)L.total, sizeof(double));
    int *N = (int *)calloc((size_t)n * n, sizeof(int));
    int rc = 0;
    memset(Nacc, 0, sizeof(long long) * (size_t)G * n * n); memset(Bacc, 0, sizeof(long long) * (size_t)G * n);
    memset(zfix, 0, sizeof(long long) * (size_t)G * n);
    for (int g = 0; g < G; g++) {
        /* the group's table spans its own observations (the engine's t_max per group) */
        double tmax = 0.0;
        for (long k = 0; k < l; k++) {
            if (group[k] != g) continue;
            if (y[k] > tmax) tmax = y[k];
            if (u && censored[k] && u[k] <= 1.7976931348623157e308 && u[k] - y[k] > tmax) tmax = u[k] - y[k];
        }
        assemble(n, T + (size_t)g * n1 * n1, C + (size_t)g * n1 * n1, theta, first, TT, S, s);
        memset(tab, 0, sizeof(double) * (size_t)L.total);
        pho_unif_table(n, S, s, pi, tmax, cap, tab);
        unif_model(n, S, s, scale, cum);
        long long *Ng = Nacc + (size_t)g * n * n, *Bg = Bacc + (size_t)g * n, *zg = zfix + (size_t)g * n;
        for (long k = 0; k < l; k++) {
            if (group[k] != g) continue;
            pht_stream st = stream_for(seed, iter, (uint32_t)k);
            memset(N, 0, sizeof(int) * (size_t)n * n);
            pho_unif_ctx ctx; ctx.N = N; ctx.n = n;
            int B = 0;
            rc |= pht_unif_path(tab, n, cap, s, scale, cum, pi, y[k], censored[k], u ? u[k] : INFINITY, &st, z, zb, 1, &ctx, &B);
            Bg[B]++;
            for (int c = 0; c < n * n; c++) Ng[c] += N[c];
            for (int i = 0; i < n; i++) if (z[i] != 0.0) zg[i] += llrint(z[i] * zs);
        }
    }
    free(pi); free(TT); free(S); free(s); free(scale); free(cum); free(zb); free(z); free(tab); free(N);
    return rc;
}

int pho_groups_update(uint64_t seed, uint32_t iter, int n, int m, int G, const double *nu, const double *zeta, const int *T,
                      const double *C, int zbits, const long long *Nacc, const long long *zfix, double *theta_new) {
    const int n1 = n + 1;
    const double zscale = ldexp(1.0, -zbits);
    for (int v = 0; v < m; v++) {
        long long Nsum = 0; double zsum = 0.0;
        for (int g = 0; g < G; g++) {
            const int *Tg = T + (size_t)g * n1 * n1; const double *Cg = C + (size_t)g * n1 * n1;
            const long long *Ng = Nacc + (size_t)g * n * n, *zg = zfix + (size_t)g * n;
            for (int i = n; i >= 0; i--)
                for (int j = n; j >= 0; j--) {
                    if (Tg[i + j * n1] != v + 1) continue;
                    Nsum += (j == n) ? Ng[i + i * n] : Ng[i + j * n];
                    const double zi = (double)zg[i] * zscale;
                    zsum += zi / Cg[i + j * n1];
                }
        }
        theta_new[v] = pho_rgamma_at(seed, iter, (uint32_t)v, nu[v] + (double)Nsum, 1.0 / (zeta[v] + zsum));
    }
    return 0;
}
