/*
 * pht_unif.h -- the uniformisation path sampler (method 64, Hobolth & Stone 2009, section 3.3), shared by the CUDA
 * kernels of k_unif.cu and the host restatement oracle/pht_oracle_unif.c, as pht_eigen.h is shared by k_model.cu and
 * the host solver.  Only IEEE add/mul/div, sqrt and pht_exp/pht_log are used, in a fixed order; host code is built
 * with -ffp-contract=off and device code with -fmad=false, so both builds give the same bits.
 *
 * Law.  With lambda = max_i (-S_ii), R = I + S/lambda (non-negative, sub-stochastic) and r = s/lambda,
 *     e^{Sx} = sum_k Pois(k; lambda x) R^k.
 * The absorbing column of the full chain [[R, r], [0, 1]]^k is g_k = 1 - R^k 1; it is tabulated as
 * g_{k+1} = r + R g_k (non-negative terms only), so no probability is ever formed by cancellation.
 *
 * Table (per sweep, one buffer, offsets from pht_unif_layout): a header (lambda, K_sweep, number of positive entries of
 * pi, the first of them), log k! (filled once per engine), R, r, then for k = 0 .. K_sweep
 *     P_k = R^k       (column-major n x n; (R^{k+1})_ij = sum_l (R^k)_il R_lj, l ascending)
 *     q_k = pi R^k    ((q_{k+1})_j = sum_l (q_k)_l R_lj, l ascending)
 *     g_k             ((g_{k+1})_i = r_i + sum_l R_il (g_k)_l, l ascending)
 *
 * Truncation.  The sums over k run to K(x) = ceil(x + 10 sqrt(x) + 20) at Poisson mean x.  The neglected tail
 * P(Pois(x) > K(x)) is below 1e-15 for every x the table admits (K(x) < PHT_UNIF_CAP, i.e. x up to ~3484; checked in
 * tests/test_unif_oracle.py).  An observation with K(x) >= capacity raises error bit 256 instead.
 *
 * Per observation, on Philox sub-stream 0 of (sweep, global observation), with x = lambda y, the draws in this order:
 *   1. b, the state at y, from (pi e^{Sy})_b times s_b (exact), 1 (right-censored) or 1 - (e^{S(u-y)} 1)_b (interval);
 *   2. a, the start state, from pi_a (e^{Sy})_ab -- only when pi has more than one positive entry and y > 0;
 *   3. (y > 0) the event count k of the bridge a -> b on [0, y], from Pois(k; x) (R^k)_ab;
 *   4. for each event i = 1..k: the spacing before it, then (i < k) the state after it, from R_{x_{i-1} c} (R^{k-i})_cb;
 *      then the last spacing.  The k+1 spacings of k uniform points on [0, y] are y E_i / sum E with E_i iid Exp(1),
 *      so the unnormalised E are summed per state and scaled once;
 *   5. exact: absorption from b at y.  Right-censored: the unconditioned chain from b (rexp with `scale`, scan of the
 *      Pfull running sums `cum`).  Interval (y, u]: a bridge of the full chain from b to absorption over [0, u - y]:
 *      event count k2 >= 1 from Pois(k2; lambda (u-y)) (g_{k2})_b, then per event its spacing and, until absorption,
 *      the next state from R_{x c} (g_{k2-i})_c (c < n) or r_x (absorption), then the last spacing.
 * Virtual self-jumps add nothing to N; an absorption from state j is counted as N[j, j] (the engine's exit marker).
 * Categorical draws take the smallest category with a positive weight whose running sum reaches U x total.
 */
#ifndef PHT_UNIF_H
#define PHT_UNIF_H

#include "pht_philox.h"

#define PHT_UNIF_CAP 4096            /* powers R^0 .. R^{cap-1} a table holds */
#define PHT_UNIF_ERR_TABLE 256       /* error word: an observation (or the sweep) needs more powers than the table holds */
#define PHT_UNIF_ERR_ZERO 512        /* error word: every weight of a draw underflowed to zero */

typedef struct { int lgk, R, r, P, q, g, total; } pht_unif_layout;

PHT_HD pht_unif_layout pht_unif_layout_make(int n, int cap) {
    pht_unif_layout L; int o = 8;            /* header: lambda, K_sweep, positive entries of pi, the first of them */
    L.lgk = o; o += cap;
    L.R = o; o += n * n;
    L.r = o; o += n;
    L.P = o; o += cap * n * n;
    L.q = o; o += cap * n;
    L.g = o; o += cap * n;
    L.total = o;
    return L;
}

/* the truncation point at Poisson mean x; a huge value for x beyond any table */
PHT_HD int pht_unif_K(double x) {
    if (!(x <= 1.0e7)) return 0x7fffffff;
    const double v = x + 10.0 * PHT_SQRT(x) + 20.0;
    int k = (int)v;
    if ((double)k < v) k++;
    return k;
}

/* Pois(k; x) = exp(k log x - x - log k!) (lx = log x); at x = 0 the point mass at k = 0 */
PHT_HD double pht_unif_w(double x, double lx, int k, const double *lgk) {
    if (x == 0.0) return k == 0 ? 1.0 : 0.0;
    return pht_exp((double)k * lx - x - lgk[k]);
}

PHT_HD void pht_unif_lgk_fill(double *lgk, int cap) {
    double acc = 0.0; lgk[0] = 0.0;
    for (int k = 1; k < cap; k++) { acc = acc + pht_log((double)k); lgk[k] = acc; }
}

PHT_HD double pht_unif_lambda(int n, const double *S) {
    double lam = 0.0;
    for (int i = 0; i < n; i++) if (-S[i + i * n] > lam) lam = -S[i + i * n];
    return lam;
}
PHT_HD double pht_unif_R_entry(int n, const double *S, double lam, int i, int j) {
    return i == j ? 1.0 + S[i + i * n] / lam : S[i + j * n] / lam;
}
/* one entry of the next power: (Pk R)_ij, q_k R at j, r + R g_k at i */
PHT_HD double pht_unif_P_entry(int n, const double *Pk, const double *R, int i, int j) {
    double acc = 0.0;
    for (int l = 0; l < n; l++) acc += Pk[i + l * n] * R[l + j * n];
    return acc;
}
PHT_HD double pht_unif_q_entry(int n, const double *qk, const double *R, int j) {
    double acc = 0.0;
    for (int l = 0; l < n; l++) acc += qk[l] * R[l + j * n];
    return acc;
}
PHT_HD double pht_unif_g_entry(int n, const double *gk, const double *R, const double *r, int i) {
    double acc = r[i];
    for (int l = 0; l < n; l++) acc += R[i + l * n] * gk[l];
    return acc;
}

/* categorical draw over w[0], w[ws], ... w[(n-1) ws]: the smallest c with w_c > 0 whose running sum reaches U x total;
 * -1 when every weight is zero */
PHT_HD int pht_unif_pick(const double *w, int n, int ws, double U) {
    double tot = 0.0;
    for (int c = 0; c < n; c++) tot += w[c * ws];
    if (!(tot > 0.0)) return -1;
    const double target = U * tot;
    double sofar = 0.0; int last = -1;
    for (int c = 0; c < n; c++) {
        const double v = w[c * ws];
        if (v > 0.0) { sofar += v; last = c; if (sofar >= target) return c; }
    }
    return last;
}

/* Delayed entry (left truncation; pht_engine_set_entry).  A unit seen only because it survived to its entry age a > 0
 * contributes L / S(a).  The augmentation of Dempster, Laird & Rubin (1977) keeps the sweep conjugate: per truncated
 * observation, M units of the same kind lost before a ("ghosts"), M | theta ~ Geometric with P(M = k) = F(a)^k S(a),
 * F = 1 - S, and each ghost's whole path given absorption in (0, a] -- the left-censored path (y = 0, u = a) of
 * pht_unif_path.  Summing F(a)^M over M gives 1 / S(a), so the theta-marginal is prior x prod L_i / S(a_i).
 * Entry tables (a buffer of their own, 2 x capacity doubles, filled per sweep for k <= K_sweep; a <= y, so K_sweep
 * covers lambda a):
 *     sigma_k = sum_c (q_k)_c           S(a) = sum_k Pois(k; lambda a) sigma_k
 *     phi_k   = sum_c pi_c (g_k)_c      F(a) = sum_k Pois(k; lambda a) phi_k
 * both sums of non-negative terms, c ascending, so neither probability is formed by cancellation.
 * Draw order, per observation with a > 0: the ghost count is draw 0 of Philox sub-stream 1 of (sweep, global
 * observation), M = floor(log U / log F(a)) with log F = log F (F <= 1/2) or log1p(-S) (otherwise); ghost j (0-based)
 * is pht_unif_path(y = 0, censored, u = a) on sub-stream 2 + j.  The observation's own path stays on sub-stream 0. */
#define PHT_UNIF_ERR_ENTRY 1024      /* error word: S(a) underflowed, or a ghost count above PHT_UNIF_GHOST_MAX */
#define PHT_UNIF_GHOST_MAX (1 << 20)

PHT_HD double pht_unif_sigma_entry(int n, const double *qk) {
    double acc = 0.0;
    for (int c = 0; c < n; c++) acc += qk[c];
    return acc;
}
PHT_HD double pht_unif_phi_entry(int n, const double *pi, const double *gk) {
    double acc = 0.0;
    for (int c = 0; c < n; c++) acc += pi[c] * gk[c];
    return acc;
}

/* The ghost count of an observation with entry age a > 0.  tab: the sweep's table; etab: sigma_k at k, phi_k at
 * cap + k; U: draw 0 of sub-stream 1.  Returns 0 or an error bit; *M = 0 on error. */
PHT_HD int pht_unif_ghost_count(const double *tab, const double *etab, int n, int cap, double a, double U, unsigned *M) {
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    const double *lgk = tab + L.lgk;
    const double x = tab[0] * a, lx = x > 0.0 ? pht_log(x) : 0.0;
    const int K = pht_unif_K(x);
    *M = 0u;
    if (K >= cap) return PHT_UNIF_ERR_TABLE;
    double S = 0.0, F = 0.0;
    for (int k = 0; k <= K; k++) {
        const double w = pht_unif_w(x, lx, k, lgk);
        if (w == 0.0) continue;
        S += w * etab[k];
        F += w * etab[cap + k];
    }
    if (!(S > 0.0)) return PHT_UNIF_ERR_ENTRY;
    const double lF = F <= 0.5 ? pht_log(F) : pht_log1p(-S);      /* < 0; -inf when F = 0 (then M = 0) */
    const double q = pht_log(U) / lF;
    if (!(q < 2.0 * PHT_UNIF_GHOST_MAX)) return PHT_UNIF_ERR_ENTRY;
    const unsigned m = (unsigned)q;
    if (m > (unsigned)PHT_UNIF_GHOST_MAX) return PHT_UNIF_ERR_ENTRY;
    *M = m;
    return 0;
}

/* the sampler itself is compiled where the includer says how transitions are counted: PHT_UNIF_CTX (a type) and
 * PHT_UNIF_COUNT(ctx, from, to); PHT_UNIF_U01(st) may replace the uniform draw by an equivalent call, PHT_UNIF_FN the function's qualifiers */
#if defined(PHT_UNIF_CTX) && defined(PHT_UNIF_COUNT)
#ifndef PHT_UNIF_U01
#define PHT_UNIF_U01(st) pht_stream_unif(st)
#endif
#ifndef PHT_UNIF_FN
#define PHT_UNIF_FN PHT_HD
#endif

/* One observation.  tab: the sweep's table; s, scale, cum, pi: the model's exit rates, rexp scales, Pfull running sums
 * ((n+1) x (n+1), row j at j (n+1)) and start distribution; u = +inf: no upper bound.  za, zb: two n-vectors of
 * scratch with stride zs; on return za holds the path's sojourn totals.  Transitions go to PHT_UNIF_COUNT(ctx, from,
 * to), the start state to *B.  Returns 0 or an error bit. */
PHT_UNIF_FN int pht_unif_path(const double *tab, int n, int cap, const double *s, const double *scale, const double *cum,
                         const double *pi, double y, int cens, double u, pht_stream *st, double *za, double *zb, int zs,
                         PHT_UNIF_CTX *ctx, int *B) {
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    const double lam = tab[0];
    const int npos = (int)tab[2], a1 = (int)tab[3];
    const double *lgk = tab + L.lgk, *R = tab + L.R, *r = tab + L.r;
    const int iv = cens && u <= 1.7976931348623157e308;
    const double x = lam * y, lx = x > 0.0 ? pht_log(x) : 0.0;
    const double d = iv ? u - y : 0.0, x2 = lam * d, lx2 = x2 > 0.0 ? pht_log(x2) : 0.0;
    const int K1 = pht_unif_K(x), K2 = iv ? pht_unif_K(x2) : 0;
    *B = 0;
    if (K1 >= cap || K2 >= cap) return PHT_UNIF_ERR_TABLE;

    /* 1. the state at y */
    for (int c = 0; c < n; c++) za[c * zs] = 0.0;
    for (int k = 0; k <= K1; k++) {
        const double w = pht_unif_w(x, lx, k, lgk);
        if (w == 0.0) continue;
        const double *q = tab + L.q + k * n;
        for (int c = 0; c < n; c++) za[c * zs] += w * q[c];
    }
    if (iv) {
        for (int c = 0; c < n; c++) zb[c * zs] = 0.0;
        for (int k = 1; k <= K2; k++) {
            const double w = pht_unif_w(x2, lx2, k, lgk);
            if (w == 0.0) continue;
            const double *g = tab + L.g + k * n;
            for (int c = 0; c < n; c++) zb[c * zs] += w * g[c];
        }
        for (int c = 0; c < n; c++) za[c * zs] = za[c * zs] * zb[c * zs];
    } else if (!cens) {
        for (int c = 0; c < n; c++) za[c * zs] = za[c * zs] * s[c];
    }
    const int b = pht_unif_pick(za, n, zs, PHT_UNIF_U01(st));
    if (b < 0) return PHT_UNIF_ERR_ZERO;

    /* 2. the start state */
    int a;
    if (y > 0.0 && npos > 1) {
        for (int c = 0; c < n; c++) za[c * zs] = 0.0;
        for (int k = 0; k <= K1; k++) {
            const double w = pht_unif_w(x, lx, k, lgk);
            if (w == 0.0) continue;
            const double *P = tab + L.P + k * n * n + b * n;
            for (int c = 0; c < n; c++) za[c * zs] += w * P[c];
        }
        for (int c = 0; c < n; c++) za[c * zs] = pi[c] * za[c * zs];
        a = pht_unif_pick(za, n, zs, PHT_UNIF_U01(st));
        if (a < 0) return PHT_UNIF_ERR_ZERO;
    } else a = y > 0.0 ? a1 : b;
    *B = a;
    for (int c = 0; c < n; c++) { za[c * zs] = 0.0; zb[c * zs] = 0.0; }

    /* 3.-4. the bridge a -> b on [0, y] */
    if (y > 0.0) {
        double tot = 0.0;
        for (int k = 0; k <= K1; k++) tot += pht_unif_w(x, lx, k, lgk) * tab[L.P + k * n * n + a + b * n];
        if (!(tot > 0.0)) return PHT_UNIF_ERR_ZERO;
        const double target = PHT_UNIF_U01(st) * tot;
        double sofar = 0.0; int kk = -1;
        for (int k = 0; k <= K1; k++) {
            const double v = pht_unif_w(x, lx, k, lgk) * tab[L.P + k * n * n + a + b * n];
            if (v > 0.0) { sofar += v; kk = k; if (sofar >= target) break; }
        }
        int cur = a; double et = 0.0;
        for (int i = 1; i <= kk; i++) {
            const double e = -pht_log(PHT_UNIF_U01(st));
            za[cur * zs] += e; et += e;
            int c = b;
            if (i < kk) {
                const double *Pn = tab + L.P + (kk - i) * n * n + b * n;
                double t2 = 0.0;
                for (int q = 0; q < n; q++) t2 += R[cur + q * n] * Pn[q];
                if (!(t2 > 0.0)) return PHT_UNIF_ERR_ZERO;
                const double tg = PHT_UNIF_U01(st) * t2;
                double so = 0.0; c = -1;
                for (int q = 0; q < n; q++) {
                    const double v = R[cur + q * n] * Pn[q];
                    if (v > 0.0) { so += v; c = q; if (so >= tg) break; }
                }
            }
            if (c != cur) PHT_UNIF_COUNT(ctx, cur, c);
            cur = c;
        }
        const double e = -pht_log(PHT_UNIF_U01(st));
        za[cur * zs] += e; et += e;
        const double sc = y / et;
        for (int c = 0; c < n; c++) if (za[c * zs] != 0.0) za[c * zs] = za[c * zs] * sc;
    }

    /* 5. after y */
    if (!cens) {
        PHT_UNIF_COUNT(ctx, b, b);
    } else if (!iv) {
        int j = b;
        for (;;) {
            const double t = scale[j] * -pht_log(PHT_UNIF_U01(st));
            const double target = PHT_UNIF_U01(st);
            const double *cr = cum + j * (n + 1);
            int k = 0;
            while (k < n && cr[k] < target) k++;
            za[j * zs] += t;
            if (k < n) { PHT_UNIF_COUNT(ctx, j, k); j = k; }
            else { PHT_UNIF_COUNT(ctx, j, j); break; }
        }
    } else {
        double tot = 0.0;
        for (int k = 1; k <= K2; k++) tot += pht_unif_w(x2, lx2, k, lgk) * tab[L.g + k * n + b];
        if (!(tot > 0.0)) return PHT_UNIF_ERR_ZERO;
        const double target = PHT_UNIF_U01(st) * tot;
        double sofar = 0.0; int kk = -1;
        for (int k = 1; k <= K2; k++) {
            const double v = pht_unif_w(x2, lx2, k, lgk) * tab[L.g + k * n + b];
            if (v > 0.0) { sofar += v; kk = k; if (sofar >= target) break; }
        }
        int cur = b, absorbed = 0; double et = 0.0;
        for (int i = 1; i <= kk; i++) {
            const double e = -pht_log(PHT_UNIF_U01(st));
            et += e;
            if (absorbed) continue;
            zb[cur * zs] += e;
            const double *gn = tab + L.g + (kk - i) * n;
            double t2 = 0.0;
            for (int q = 0; q < n; q++) t2 += R[cur + q * n] * gn[q];
            t2 += r[cur];
            if (!(t2 > 0.0)) return PHT_UNIF_ERR_ZERO;
            const double tg = PHT_UNIF_U01(st) * t2;
            double so = 0.0; int c = -1;
            for (int q = 0; q < n; q++) {
                const double v = R[cur + q * n] * gn[q];
                if (v > 0.0) { so += v; c = q; if (so >= tg) break; }
            }
            if (!(so >= tg) && r[cur] > 0.0) c = n;      /* absorption: the last category */
            if (c == n) { PHT_UNIF_COUNT(ctx, cur, cur); absorbed = 1; }
            else { if (c != cur) PHT_UNIF_COUNT(ctx, cur, c); cur = c; }
        }
        const double e = -pht_log(PHT_UNIF_U01(st));
        et += e;
        const double sc = d / et;
        for (int c = 0; c < n; c++) if (zb[c * zs] != 0.0) za[c * zs] = za[c * zs] + zb[c * zs] * sc;
    }
    return 0;
}
#endif /* PHT_UNIF_CTX */

#endif /* PHT_UNIF_H */
