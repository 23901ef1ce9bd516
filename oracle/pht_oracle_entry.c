/*
 * pht_oracle_entry.c -- CPU restatement of delayed entry (left truncation) for the uniformisation sampler (method 64;
 * TEST INFRASTRUCTURE ONLY, like pht_oracle.c).  Law, draw order and arithmetic are those of
 * phasetype_b200/csrc/pht_unif.h ("Delayed entry"), built here for the host: the entry tables sigma_k and phi_k, the ghost
 * count of each observation (draw 0 of Philox sub-stream 1) and its ghost paths (left-censored on (0, a], sub-stream
 * 2 + j).  It includes pht_oracle_unif.c for the table, the observed paths and the model pieces, and sums the ghosts into
 * the same fixed point.  Built by pyoracle_entry.build() into _build/libphtoracle_entry.so, a library of its own.
 *
 *   double pho_log1p(x), pho_log1p_general(x)                 the shared log1p, fast path and general path
 *   int pho_entry_tables(n, S, s, pi, tmax, cap, etab)        -> K_sweep; sigma_k at k, phi_k at cap + k
 *   int pho_entry_paths(seed, iter, obs0, stride, count, y, cens, u, a, pi, n, S, s, cap, outM, total, outB, outN, outz)
 *   int pho_entry_sweep_stats(seed, iter, first, n, m, T, C, theta, y, l, cens, u, a, pi, rank, world, zbits, cap,
 *                             Nacc, Bacc, zfix)
 * u, pi as in pht_oracle_unif.c; outB may be NULL (counts only), else it receives total = sum M ghost paths in
 * (observation, ghost index) order.  The return value is 0 or the engine's error bits (256, 512, 1024), or -1 when
 * total does not match.
 */
#include "pht_oracle_unif.c"

double pho_log1p(double x) { return pht_log1p(x); }
double pho_log1p_general(double x) { return pht_log1p_general(x); }

static void entry_tables(int n, const double *tab, const double *pi, int cap, double *etab) {
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    const int K = (int)tab[1];
    for (int k = 0; k <= K; k++) {
        etab[k] = pht_unif_sigma_entry(n, tab + L.q + k * n);
        etab[cap + k] = pht_unif_phi_entry(n, pi, tab + L.g + k * n);
    }
}

int pho_entry_tables(int n, const double *S, const double *s, const double *pi, double tmax, int cap, double *etab) {
    double *tab = (double *)calloc((size_t)pht_unif_layout_make(n, cap).total, sizeof(double));
    const int K = pho_unif_table(n, S, s, pi, tmax, cap, tab);
    entry_tables(n, tab, pi, cap, etab);
    free(tab);
    return K;
}

int pho_entry_paths(uint64_t seed, uint32_t iter, long obs0, long stride, long count, const double *y, const int *cens,
                    const double *u, const double *a, const double *pi_in, int n, const double *S, const double *s, int cap,
                    int *outM, long total, int *outB, int *outN, double *outz) {
    double *pi = (double *)calloc(n, sizeof(double));
    if (pi_in) for (int i = 0; i < n; i++) pi[i] = pi_in[i];
    else pi[0] = 1.0;
    double tmax = 0.0;
    for (long k = 0; k < count; k++) {
        if (y[k] > tmax) tmax = y[k];
        if (u && cens[k] && u[k] <= 1.7976931348623157e308 && u[k] - y[k] > tmax) tmax = u[k] - y[k];
    }
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    double *tab = (double *)calloc((size_t)L.total, sizeof(double)), *etab = (double *)calloc((size_t)2 * cap, sizeof(double));
    double *scale = (double *)calloc(n, sizeof(double)), *cum = (double *)calloc((size_t)(n + 1) * (n + 1), sizeof(double));
    double *zb = (double *)calloc(n, sizeof(double));
    int rc = 0;
    pho_unif_table(n, S, s, pi, tmax, cap, tab);
    entry_tables(n, tab, pi, cap, etab);
    unif_model(n, S, s, scale, cum);
    long G = 0;
    for (long k = 0; k < count; k++) {
        unsigned M = 0;
        const uint32_t og = (uint32_t)(obs0 + k * stride);
        if (a[k] > 0.0)
            rc |= pht_unif_ghost_count(tab, etab, n, cap, a[k], pht_unif_at((uint32_t)seed, (uint32_t)(seed >> 32), iter, og, 1u, 0u), &M);
        outM[k] = (int)M;
        G += M;
    }
    if (outB && G != total) rc = -1;
    if (outB && rc == 0) {
        long g = 0;
        for (long k = 0; k < count; k++) {
            const uint32_t og = (uint32_t)(obs0 + k * stride);
            for (int j = 0; j < outM[k]; j++, g++) {
                pht_stream st; st.k0 = (uint32_t)seed; st.k1 = (uint32_t)(seed >> 32);
                pht_stream_seek(&st, iter, og, 2u + (uint32_t)j, 0u);
                int *N = outN + (size_t)g * n * n;
                memset(N, 0, sizeof(int) * (size_t)n * n);
                pho_unif_ctx ctx; ctx.N = N; ctx.n = n;
                rc |= pht_unif_path(tab, n, cap, s, scale, cum, pi, 0.0, 1, a[k], &st, outz + (size_t)g * n, zb, 1, &ctx, &outB[g]);
            }
        }
    }
    free(pi); free(tab); free(etab); free(scale); free(cum); free(zb);
    return rc;
}

int pho_entry_sweep_stats(uint64_t seed, uint32_t iter, int first, int n, int m, const int *T, const double *C,
                          const double *theta, const double *y, long l, const int *censored, const double *u, const double *a,
                          const double *pi, int rank, int world, int zbits, int cap, long long *Nacc, long long *Bacc, long long *zfix) {
    int rc = pho_unif_sweep_stats(seed, iter, first, n, m, T, C, theta, y, l, censored, u, pi, rank, world, zbits, cap, Nacc, Bacc, zfix);
    if (rc) return rc;
    const int n1 = n + 1;
    long cnt = 0;
    for (long i = rank; i < l; i += world) cnt++;
    double *TT = (double *)calloc((size_t)n1 * n1, sizeof(double)), *S = (double *)calloc((size_t)n * n, sizeof(double));
    double *s = (double *)calloc(n, sizeof(double));
    double *yl = (double *)malloc(sizeof(double) * (size_t)(cnt + 1)), *ul = (double *)malloc(sizeof(double) * (size_t)(cnt + 1));
    double *al = (double *)malloc(sizeof(double) * (size_t)(cnt + 1));
    int *cl = (int *)malloc(sizeof(int) * (size_t)(cnt + 1)), *M = (int *)malloc(sizeof(int) * (size_t)(cnt + 1));
    long k = 0;
    for (long i = rank; i < l; i += world, k++) { yl[k] = y[i]; cl[k] = censored[i]; ul[k] = u ? u[i] : INFINITY; al[k] = a[i]; }
    assemble(n, T, C, theta, first, TT, S, s);
    rc = pho_entry_paths(seed, iter, rank, world, cnt, yl, cl, ul, al, pi, n, S, s, cap, M, 0, NULL, NULL, NULL);
    long G = 0;
    for (k = 0; k < cnt; k++) G += M[k];
    if (rc == 0 && G > 0) {
        int *B = (int *)malloc(sizeof(int) * (size_t)G), *N = (int *)malloc(sizeof(int) * (size_t)G * n * n);
        double *z = (double *)malloc(sizeof(double) * (size_t)G * n);
        rc = pho_entry_paths(seed, iter, rank, world, cnt, yl, cl, ul, al, pi, n, S, s, cap, M, G, B, N, z);
        const double zs = ldexp(1.0, zbits);
        for (long g = 0; g < G; g++) {
            Bacc[B[g]]++;
            for (int c = 0; c < n * n; c++) Nacc[c] += N[(size_t)g * n * n + c];
            for (int i = 0; i < n; i++) { const double v = z[(size_t)g * n + i]; if (v != 0.0) zfix[i] += llrint(v * zs); }
        }
        free(B); free(N); free(z);
    }
    free(TT); free(S); free(s); free(yl); free(ul); free(al); free(cl); free(M);
    return rc;
}
