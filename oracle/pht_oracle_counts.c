/*
 * pht_oracle_counts.c -- CPU build of the record form of the uniformisation sampler (method 64 with counts; TEST
 * INFRASTRUCTURE ONLY, like pht_oracle.c): pht_unif_rec and pht_unif_rec_path of phasetype_b200/csrc/pht_unif.h, next to
 * the per-observation sampler of pht_oracle_unif.c, which it includes (table, model pieces, streams).  The reference for
 * a record of w units is the per-observation sampler on the expanded data; tests/test_counts_oracle.py compares the two.
 * Built by pyoracle_counts.build() into _build/libphtoracle_counts.so, a library of its own.
 *
 *   int pho_unif_record_paths(seed, iter, records, y, cens, u, pi, counts, n, S, s, cap, kb, outB, outN, outz)
 */
#include "pht_oracle_unif.c"

/* Per record with count w > 0: its weights, the vector of the state at y and the start-state matrix prepared by plain
 * loops over k, states and cells, then its w units on the streams of the expanded observations base + j (base: the
 * exclusive prefix sum of the counts).  Outputs in expanded order, as pho_unif_paths writes them for
 * np.repeat(records, counts); kb bounds the weight buffers (weights beyond are recomputed). */
int pho_unif_record_paths(uint64_t seed, uint32_t iter, long records, const double *y, const int *cens, const double *u,
                          const double *pi_in, const unsigned *counts, int n, const double *S, const double *s, int cap, int kb,
                          int *outB, int *outN, double *outz) {
    double *pi = (double *)calloc(n, sizeof(double));
    if (pi_in) for (int i = 0; i < n; i++) pi[i] = pi_in[i];
    else pi[0] = 1.0;
    double tmax = 0.0;
    for (long k = 0; k < records; k++) {
        if (!counts[k]) continue;
        if (y[k] > tmax) tmax = y[k];
        if (u && cens[k] && u[k] <= 1.7976931348623157e308 && u[k] - y[k] > tmax) tmax = u[k] - y[k];
    }
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    double *tab = (double *)calloc((size_t)L.total, sizeof(double));
    double *scale = (double *)calloc(n, sizeof(double)), *cum = (double *)calloc((size_t)(n + 1) * (n + 1), sizeof(double));
    double *zb = (double *)calloc(n, sizeof(double));
    double *w1 = (double *)calloc((size_t)kb + 1, sizeof(double)), *w2 = (double *)calloc((size_t)kb + 1, sizeof(double));
    double *v = (double *)calloc(n, sizeof(double)), *mx = (double *)calloc((size_t)n * n, sizeof(double));
    int rc = 0;
    pho_unif_table(n, S, s, pi, tmax, cap, tab);
    unif_model(n, S, s, scale, cum);
    const double *lgk = tab + L.lgk;
    uint64_t base = 0;
    for (long k = 0; k < records; k++) {
        if (!counts[k]) continue;
        pht_unif_rec rec;
        const int e0 = pht_unif_rec_init(&rec, tab, cap, y[k], cens[k], u ? u[k] : INFINITY, kb);
        rec.w1 = w1; rec.w2 = w2; rec.v = v; rec.mx = mx;
        if (!e0) {
            for (int j = 0; j <= rec.K1 && j <= kb; j++) w1[j] = pht_unif_w(rec.x, rec.lx, j, lgk);
            if (rec.iv) for (int j = 0; j <= rec.K2 && j <= kb; j++) w2[j] = pht_unif_w(rec.x2, rec.lx2, j, lgk);
            for (int c = 0; c < n; c++) v[c] = pht_unif_rec_v_entry(&rec, tab, n, cap, s, c);
            if (y[k] > 0.0 && (int)tab[2] > 1)
                for (int b = 0; b < n; b++) for (int c = 0; c < n; c++) mx[c + b * n] = pht_unif_rec_m_entry(&rec, tab, n, cap, pi, c, b);
        }
        for (unsigned j = 0; j < counts[k]; j++, base++) {
            pht_stream st = stream_for(seed, iter, (uint32_t)base);
            int *N = outN + (size_t)base * n * n;
            memset(N, 0, sizeof(int) * (size_t)n * n);
            pho_unif_ctx ctx; ctx.N = N; ctx.n = n;
            if (e0) { rc |= e0; outB[base] = 0; continue; }
            rc |= pht_unif_rec_path(tab, n, cap, scale, cum, &rec, &st, outz + (size_t)base * n, zb, 1, &ctx, &outB[base]);
        }
    }
    free(pi); free(tab); free(scale); free(cum); free(zb); free(w1); free(w2); free(v); free(mx);
    return rc;
}
