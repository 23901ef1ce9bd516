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

/* Records with counts (pht_engine_set_counts).  The w tied units of a record (y, flag, u) are w observations whose
 * paths differ only in their Philox streams, so everything pht_unif_path computes before its first draw is computed
 * once per record: the Poisson weights of k <= K1 (and of 1 <= k <= K2 for an interval), the n weights of the state at y,
 * and, when pi has more than one positive entry and y > 0, the n x n weights of the start state given the state at y.
 * pht_unif_rec_path then draws one unit from them.  Every quantity is the same expression, summed in the same order with
 * the same zero-weight skips, as in pht_unif_path, so a unit's path is bit for bit that observation's path.  The two
 * forms are separate code: a lane cannot hold K weights of its own, a warp preparing one record can.
 * Weight buffers hold k <= kb; weights beyond are recomputed by pht_unif_w, which gives the same bits. */
typedef struct {
    double y, u, d, x, lx, x2, lx2;
    int cens, iv, K1, K2, kb;
    const double *w1, *w2;       /* w1[k] = Pois(k; lambda y), k <= min(K1, kb); w2[k] = Pois(k; lambda (u - y)), 1 <= k <= min(K2, kb) */
    const double *v;             /* the n weights of the state at y (step 1, before the pick) */
    const double *mx;            /* column b (n x n, column-major): pi_c sum_k w1[k] (R^k)_cb (only y > 0 and npos > 1) */
} pht_unif_rec;

/* the record's scalars; 0 or PHT_UNIF_ERR_TABLE (the same test as pht_unif_path) */
PHT_HD int pht_unif_rec_init(pht_unif_rec *rc, const double *tab, int cap, double y, int cens, double u, int kb) {
    const double lam = tab[0];
    rc->y = y; rc->cens = cens; rc->u = u; rc->kb = kb;
    rc->iv = cens && u <= 1.7976931348623157e308;
    rc->x = lam * y; rc->lx = rc->x > 0.0 ? pht_log(rc->x) : 0.0;
    rc->d = rc->iv ? u - y : 0.0; rc->x2 = lam * rc->d; rc->lx2 = rc->x2 > 0.0 ? pht_log(rc->x2) : 0.0;
    rc->K1 = pht_unif_K(rc->x); rc->K2 = rc->iv ? pht_unif_K(rc->x2) : 0;
    return (rc->K1 >= cap || rc->K2 >= cap) ? PHT_UNIF_ERR_TABLE : 0;
}
PHT_HD double pht_unif_rec_w1(const pht_unif_rec *rc, int k, const double *lgk) {
    return k <= rc->kb ? rc->w1[k] : pht_unif_w(rc->x, rc->lx, k, lgk);
}
PHT_HD double pht_unif_rec_w2(const pht_unif_rec *rc, int k, const double *lgk) {
    return k <= rc->kb ? rc->w2[k] : pht_unif_w(rc->x2, rc->lx2, k, lgk);
}
/* entry c of the weights of the state at y (pht_unif_path step 1); the weight buffers must be filled */
PHT_HD double pht_unif_rec_v_entry(const pht_unif_rec *rc, const double *tab, int n, int cap, const double *s, int c) {
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    const double *lgk = tab + L.lgk;
    double v = 0.0;
    for (int k = 0; k <= rc->K1; k++) {
        const double w = pht_unif_rec_w1(rc, k, lgk);
        if (w == 0.0) continue;
        v += w * tab[L.q + k * n + c];
    }
    if (rc->iv) {
        double z = 0.0;
        for (int k = 1; k <= rc->K2; k++) {
            const double w = pht_unif_rec_w2(rc, k, lgk);
            if (w == 0.0) continue;
            z += w * tab[L.g + k * n + c];
        }
        v = v * z;
    } else if (!rc->cens) {
        v = v * s[c];
    }
    return v;
}
/* entry (c, b) of the start-state weights (pht_unif_path step 2 for state b at y) */
PHT_HD double pht_unif_rec_m_entry(const pht_unif_rec *rc, const double *tab, int n, int cap, const double *pi, int c, int b) {
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    const double *lgk = tab + L.lgk;
    double a = 0.0;
    for (int k = 0; k <= rc->K1; k++) {
        const double w = pht_unif_rec_w1(rc, k, lgk);
        if (w == 0.0) continue;
        a += w * tab[L.P + k * n * n + b * n + c];
    }
    return pi[c] * a;
}

/* Panel observations (pht_engine_set_visits).  Observation i carries visits (t_j, A_j), j = 1..m, 0 <= t_1 < ... < t_m <= y,
 * A_j a non-empty set of phases (bit c of a uint32 mask: phase c).  The path law is that of the absorbing chain given pi,
 * the visits and the terminal information: a hidden Markov chain over the visit states, each gap a bridge with fixed ends.
 * Backward pass (no draws), with t_0 = 0 and d_{m+1} = y - t_m:
 *     v = s (exact), 1 (right-censored) or sum_{k>=1} Pois(k; lambda (u - y)) g_k (interval, as in pht_unif_path step 1),
 *     beta_m = 1[A_m] . e^{S d_{m+1}} v,   beta_{j-1} = 1[A_{j-1}] . e^{S (t_j - t_{j-1})} beta_j,   beta_0 = e^{S t_1} beta_1
 * (no mask on beta_0; t_1 = 0 makes it beta_1 itself), every e^{Sd} w as sum_{k <= K(lambda d)} Pois(k; lambda d) R^k w with
 * the zero-weight skip of pht_unif_path, k ascending, then the entries of R^k w in column order.  Each beta is scaled by the
 * power of two that brings its largest entry into [1, 2): exact, and no draw depends on it, so a long panel cannot
 * underflow.  The draws, all on Philox sub-stream 0 of (sweep, global observation), in this order:
 *   1. a, the start state, from pi_a beta_0(a) -- only when pi has more than one positive entry (else the first of them);
 *   2. for j = 1..m the visit state x_j from (e^{S(t_j - t_{j-1})})_{x_{j-1} x} beta_j(x) (x_0 = a); a gap of length 0
 *      (t_1 = 0) gives x_1 = a and a one-phase mask its phase, neither with a draw;
 *   3. b, the state at y, from (e^{S d_{m+1}})_{x_m b} v_b (pht_unif_path step 1 with row x_m of R^k in place of q_k);
 *      none when t_m = y (b = x_m);
 *   4. the bridges x_0 -> x_1, ..., x_{m-1} -> x_m, x_m -> b in time order, each with the event-count / spacing /
 *      next-state draws of pht_unif_path steps 3-4 and its spacings scaled to its own length; a gap of length 0 draws
 *      nothing;
 *   5. step 5 of pht_unif_path from b.
 * B is the start state a.  Sub-streams 1 and 2 + j stay the ghosts' (delayed entry).  Every gap is at most y, so the
 * sweep's table covers it.  Scratch: (m + 1) n doubles of beta per observation (entry c of beta_j at (j n + c) bs). */

/* out = e^{S d} w (x = lambda d, lx = log x, K = K(x)); w and out may not overlap */
PHT_HD void pht_unif_expv(const double *tab, int n, int cap, double x, double lx, int K, const double *w, long ws, double *out, long os) {
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    const double *lgk = tab + L.lgk;
    for (int c = 0; c < n; c++) out[c * os] = 0.0;
    for (int k = 0; k <= K; k++) {
        const double p = pht_unif_w(x, lx, k, lgk);
        if (p == 0.0) continue;
        const double *P = tab + L.P + k * n * n;
        for (int c = 0; c < n; c++) {
            double acc = 0.0;
            for (int e = 0; e < n; e++) acc += P[c + e * n] * w[e * ws];
            out[c * os] += p * acc;
        }
    }
}

/* row a of e^{S d} (x = lambda d): out_c = sum_k Pois(k; x) (R^k)_ac, k ascending with the zero-weight skip */
PHT_HD void pht_unif_exprow(const double *tab, int n, int cap, double x, double lx, int K, int a, double *out, int os) {
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    const double *lgk = tab + L.lgk;
    for (int c = 0; c < n; c++) out[c * os] = 0.0;
    for (int k = 0; k <= K; k++) {
        const double p = pht_unif_w(x, lx, k, lgk);
        if (p == 0.0) continue;
        const double *P = tab + L.P + k * n * n + a;
        for (int c = 0; c < n; c++) out[c * os] += p * P[c * n];
    }
}

/* scale w (mask bits clear: zero) by the power of two that brings its largest entry into [1, 2); 0 or PHT_UNIF_ERR_ZERO */
PHT_HD int pht_unif_rescale(double *w, long ws, int n, uint32_t mask) {
    double mx = 0.0;
    for (int c = 0; c < n; c++) {
        if (!((mask >> c) & 1u)) w[c * ws] = 0.0;
        else if (w[c * ws] > mx) mx = w[c * ws];
    }
    if (!(mx > 0.0)) return PHT_UNIF_ERR_ZERO;
    int ex = (int)((pht_d2u(mx) >> 52) & 0x7ff);
    if (ex < 1) ex = 1;
    if (ex > 2045) ex = 2045;
    const double sc = pht_u2d((uint64_t)(2046 - ex) << 52);      /* 2^(1023 - ex) */
    for (int c = 0; c < n; c++) w[c * ws] = w[c * ws] * sc;
    return 0;
}

/* Misclassified panel observations (pht_engine_set_stage_visits).  Visit j records an observed stage o_j in 0..S-1 instead
 * of a mask, read through the emission matrix E (n x S, row-major): P(stage o read | phase c) = E[c S + o].  The law is
 * that of panel observations with the indicator 1[A_j] replaced by the emission column E[., o_j]:
 *     beta_m = E[., o_m] . e^{S d_{m+1}} v,   beta_{j-1} = E[., o_{j-1}] . e^{S (t_j - t_{j-1})} beta_j,
 * each beta rescaled by pht_unif_rescale with the mask set to the support of its column.  The draws and their order are
 * those of pht_unif_panel_path (steps 1-5), a visit state drawn only when the column's support has more than one phase
 * and the gap is not 0.  With E the 0/1 indicator of a partition into stages, every weight is the mask form's weight
 * (multiplying by 1.0 and zeroing outside the support are exact), so the paths are bit for bit those of the masks.
 * Each drawn visit state x_j is left in entry 0 of beta_j, where the caller counts K[x_j S + o_j] for E's update. */

/* the support of column o of E (n x S, row-major) as a phase mask */
PHT_HD uint32_t pht_unif_col_support(const double *E, int n, int S, uint32_t o) {
    uint32_t mk = 0u;
    for (int c = 0; c < n; c++) if (E[c * S + (int)o] > 0.0) mk |= 1u << c;
    return mk;
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

/* One unit of a prepared record (pht_unif_rec: scalars, weight buffers, rc->v and, when y > 0 and pi has more than one
 * positive entry, rc->mx): the draws of pht_unif_path from the same stream, with the same results.  Arguments as there. */
PHT_UNIF_FN int pht_unif_rec_path(const double *tab, int n, int cap, const double *scale, const double *cum,
                                  const pht_unif_rec *rc, pht_stream *st, double *za, double *zb, int zs, PHT_UNIF_CTX *ctx, int *B) {
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    const int npos = (int)tab[2], a1 = (int)tab[3];
    const double *lgk = tab + L.lgk, *R = tab + L.R, *r = tab + L.r;
    const double y = rc->y, d = rc->d;
    const int cens = rc->cens, iv = rc->iv, K1 = rc->K1, K2 = rc->K2;
    *B = 0;

    /* 1.-2. the state at y and the start state from the record's weights */
    const int b = pht_unif_pick(rc->v, n, 1, PHT_UNIF_U01(st));
    if (b < 0) return PHT_UNIF_ERR_ZERO;
    int a;
    if (y > 0.0 && npos > 1) {
        a = pht_unif_pick(rc->mx + b * n, n, 1, PHT_UNIF_U01(st));
        if (a < 0) return PHT_UNIF_ERR_ZERO;
    } else a = y > 0.0 ? a1 : b;
    *B = a;
    for (int c = 0; c < n; c++) { za[c * zs] = 0.0; zb[c * zs] = 0.0; }

    /* 3.-4. the bridge a -> b on [0, y] */
    if (y > 0.0) {
        double tot = 0.0;
        for (int k = 0; k <= K1; k++) tot += pht_unif_rec_w1(rc, k, lgk) * tab[L.P + k * n * n + a + b * n];
        if (!(tot > 0.0)) return PHT_UNIF_ERR_ZERO;
        const double target = PHT_UNIF_U01(st) * tot;
        double sofar = 0.0; int kk = -1;
        for (int k = 0; k <= K1; k++) {
            const double v = pht_unif_rec_w1(rc, k, lgk) * tab[L.P + k * n * n + a + b * n];
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
        for (int k = 1; k <= K2; k++) tot += pht_unif_rec_w2(rc, k, lgk) * tab[L.g + k * n + b];
        if (!(tot > 0.0)) return PHT_UNIF_ERR_ZERO;
        const double target = PHT_UNIF_U01(st) * tot;
        double sofar = 0.0; int kk = -1;
        for (int k = 1; k <= K2; k++) {
            const double v = pht_unif_rec_w2(rc, k, lgk) * tab[L.g + k * n + b];
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

/* A bridge a -> b over a gap of length d > 0 (x = lambda d, K = K(x)): the draws of pht_unif_path steps 3-4.  Its sojourns
 * (spacings scaled to d) are added to za; zb is scratch that is left zero. */
PHT_UNIF_FN int pht_unif_bridge(const double *tab, int n, int cap, double d, double x, double lx, int K, int a, int b,
                                pht_stream *st, double *za, double *zb, int zs, PHT_UNIF_CTX *ctx) {
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    const double *lgk = tab + L.lgk, *R = tab + L.R;
    double tot = 0.0;
    for (int k = 0; k <= K; k++) tot += pht_unif_w(x, lx, k, lgk) * tab[L.P + k * n * n + a + b * n];
    if (!(tot > 0.0)) return PHT_UNIF_ERR_ZERO;
    const double target = PHT_UNIF_U01(st) * tot;
    double sofar = 0.0; int kk = -1;
    for (int k = 0; k <= K; k++) {
        const double v = pht_unif_w(x, lx, k, lgk) * tab[L.P + k * n * n + a + b * n];
        if (v > 0.0) { sofar += v; kk = k; if (sofar >= target) break; }
    }
    int cur = a; double et = 0.0;
    for (int i = 1; i <= kk; i++) {
        const double e = -pht_log(PHT_UNIF_U01(st));
        zb[cur * zs] += e; et += e;
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
    zb[cur * zs] += e; et += e;
    const double sc = d / et;
    for (int c = 0; c < n; c++) if (zb[c * zs] != 0.0) { za[c * zs] = za[c * zs] + zb[c * zs] * sc; zb[c * zs] = 0.0; }
    return 0;
}

/* Twin: pht_unif_emis_path below repeats this function with emission columns; a fix to one belongs in the other.
 * One panel observation (law and draw order above): m >= 1 visits at times vt[0..m-1] with masks vm[0..m-1]; beta:
 * (m + 1) n doubles of scratch with stride bs.  Other arguments as pht_unif_path. */
PHT_UNIF_FN int pht_unif_panel_path(const double *tab, int n, int cap, const double *s, const double *scale, const double *cum,
                                    const double *pi, double y, int cens, double u, int m, const double *vt, const uint32_t *vm,
                                    double *beta, long bs, pht_stream *st, double *za, double *zb, int zs, PHT_UNIF_CTX *ctx, int *B) {
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    const double lam = tab[0];
    const int npos = (int)tab[2], a1 = (int)tab[3];
    const double *lgk = tab + L.lgk, *R = tab + L.R, *r = tab + L.r;
    const int iv = cens && u <= 1.7976931348623157e308;
    const double d = iv ? u - y : 0.0, x2 = lam * d, lx2 = x2 > 0.0 ? pht_log(x2) : 0.0;
    const int K2 = iv ? pht_unif_K(x2) : 0;
    const double dy = y - vt[m - 1];
    *B = 0;
    if (pht_unif_K(lam * y) >= cap || K2 >= cap) return PHT_UNIF_ERR_TABLE;
#define PHT_BETA(j, c) beta[((long)(j) * n + (c)) * bs]

    /* terminal weights v (into za) and the backward pass */
    if (iv) {
        for (int c = 0; c < n; c++) za[c * zs] = 0.0;
        for (int k = 1; k <= K2; k++) {
            const double w = pht_unif_w(x2, lx2, k, lgk);
            if (w == 0.0) continue;
            const double *g = tab + L.g + k * n;
            for (int c = 0; c < n; c++) za[c * zs] += w * g[c];
        }
    } else for (int c = 0; c < n; c++) za[c * zs] = cens ? 1.0 : s[c];
    for (int j = m; j >= 0; j--) {
        const double gap = j == m ? dy : vt[j] - (j > 0 ? vt[j - 1] : 0.0);
        const double x = lam * gap, lx = x > 0.0 ? pht_log(x) : 0.0;
        if (j == m) pht_unif_expv(tab, n, cap, x, lx, pht_unif_K(x), za, zs, &PHT_BETA(j, 0), bs);
        else pht_unif_expv(tab, n, cap, x, lx, pht_unif_K(x), &PHT_BETA(j + 1, 0), bs, &PHT_BETA(j, 0), bs);
        if (pht_unif_rescale(&PHT_BETA(j, 0), bs, n, j > 0 ? vm[j - 1] : 0xffffffffu)) return PHT_UNIF_ERR_ZERO;
    }

    /* 1. the start state */
    int a;
    if (npos > 1) {
        for (int c = 0; c < n; c++) za[c * zs] = pi[c] * PHT_BETA(0, c);
        a = pht_unif_pick(za, n, zs, PHT_UNIF_U01(st));
        if (a < 0) return PHT_UNIF_ERR_ZERO;
    } else {
        a = a1;
        if (!(PHT_BETA(0, a) > 0.0)) return PHT_UNIF_ERR_ZERO;
    }
    *B = a;

    /* 2. the visit states; x_j replaces beta_j(0), which no later draw reads */
    int prev = a;
    for (int j = 1; j <= m; j++) {
        const double gap = vt[j - 1] - (j > 1 ? vt[j - 2] : 0.0);
        const uint32_t mk = vm[j - 1];
        int x;
        if (gap == 0.0) x = prev;
        else if ((mk & (mk - 1u)) == 0u) { x = 0; while (!((mk >> x) & 1u)) x++; }
        else {
            const double xx = lam * gap;
            pht_unif_exprow(tab, n, cap, xx, xx > 0.0 ? pht_log(xx) : 0.0, pht_unif_K(xx), prev, za, zs);
            for (int c = 0; c < n; c++) za[c * zs] = za[c * zs] * PHT_BETA(j, c);
            x = pht_unif_pick(za, n, zs, PHT_UNIF_U01(st));
            if (x < 0) return PHT_UNIF_ERR_ZERO;
        }
        PHT_BETA(j, 0) = (double)x;
        prev = x;
    }

    /* 3. the state at y */
    int b = prev;
    if (dy > 0.0) {
        const double xx = lam * dy;
        pht_unif_exprow(tab, n, cap, xx, xx > 0.0 ? pht_log(xx) : 0.0, pht_unif_K(xx), prev, za, zs);
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
        b = pht_unif_pick(za, n, zs, PHT_UNIF_U01(st));
        if (b < 0) return PHT_UNIF_ERR_ZERO;
    }
    for (int c = 0; c < n; c++) { za[c * zs] = 0.0; zb[c * zs] = 0.0; }

    /* 4. the bridges in time order */
    prev = a;
    for (int j = 1; j <= m + 1; j++) {
        const double gap = j > m ? dy : vt[j - 1] - (j > 1 ? vt[j - 2] : 0.0);
        const int x = j > m ? b : (int)PHT_BETA(j, 0);
        if (gap > 0.0) {
            const double xx = lam * gap;
            const int e = pht_unif_bridge(tab, n, cap, gap, xx, xx > 0.0 ? pht_log(xx) : 0.0, pht_unif_K(xx), prev, x, st, za, zb, zs, ctx);
            if (e) return e;
        }
        prev = x;
    }
#undef PHT_BETA

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
/* Twin of pht_unif_panel_path above (kept apart so that its code and SASS stay as they are); a fix to one belongs in the
 * other.  One misclassified panel observation (law above "Misclassified panel observations"): m >= 1 visits at times vt[0..m-1]
 * with observed stages vo[0..m-1], read through E (n x S, row-major); beta: (m + 1) n doubles of scratch with stride bs,
 * entry 0 of beta_j holding the drawn x_j on return.  Other arguments as pht_unif_panel_path. */
PHT_UNIF_FN int pht_unif_emis_path(const double *tab, int n, int cap, const double *s, const double *scale, const double *cum,
                                   const double *pi, double y, int cens, double u, int m, const double *vt, const uint32_t *vo,
                                   const double *E, int S, double *beta, long bs, pht_stream *st, double *za, double *zb, int zs,
                                   PHT_UNIF_CTX *ctx, int *B) {
    const pht_unif_layout L = pht_unif_layout_make(n, cap);
    const double lam = tab[0];
    const int npos = (int)tab[2], a1 = (int)tab[3];
    const double *lgk = tab + L.lgk, *R = tab + L.R, *r = tab + L.r;
    const int iv = cens && u <= 1.7976931348623157e308;
    const double d = iv ? u - y : 0.0, x2 = lam * d, lx2 = x2 > 0.0 ? pht_log(x2) : 0.0;
    const int K2 = iv ? pht_unif_K(x2) : 0;
    const double dy = y - vt[m - 1];
    *B = 0;
    if (pht_unif_K(lam * y) >= cap || K2 >= cap) return PHT_UNIF_ERR_TABLE;
#define PHT_BETA(j, c) beta[((long)(j) * n + (c)) * bs]

    /* terminal weights v (into za) and the backward pass */
    if (iv) {
        for (int c = 0; c < n; c++) za[c * zs] = 0.0;
        for (int k = 1; k <= K2; k++) {
            const double w = pht_unif_w(x2, lx2, k, lgk);
            if (w == 0.0) continue;
            const double *g = tab + L.g + k * n;
            for (int c = 0; c < n; c++) za[c * zs] += w * g[c];
        }
    } else for (int c = 0; c < n; c++) za[c * zs] = cens ? 1.0 : s[c];
    for (int j = m; j >= 0; j--) {
        const double gap = j == m ? dy : vt[j] - (j > 0 ? vt[j - 1] : 0.0);
        const double x = lam * gap, lx = x > 0.0 ? pht_log(x) : 0.0;
        if (j == m) pht_unif_expv(tab, n, cap, x, lx, pht_unif_K(x), za, zs, &PHT_BETA(j, 0), bs);
        else pht_unif_expv(tab, n, cap, x, lx, pht_unif_K(x), &PHT_BETA(j + 1, 0), bs, &PHT_BETA(j, 0), bs);
        uint32_t mk = 0xffffffffu;
        if (j > 0) {
            const uint32_t o = vo[j - 1];
            mk = pht_unif_col_support(E, n, S, o);
            for (int c = 0; c < n; c++) PHT_BETA(j, c) = PHT_BETA(j, c) * E[c * S + (int)o];
        }
        if (pht_unif_rescale(&PHT_BETA(j, 0), bs, n, mk)) return PHT_UNIF_ERR_ZERO;
    }

    /* 1. the start state */
    int a;
    if (npos > 1) {
        for (int c = 0; c < n; c++) za[c * zs] = pi[c] * PHT_BETA(0, c);
        a = pht_unif_pick(za, n, zs, PHT_UNIF_U01(st));
        if (a < 0) return PHT_UNIF_ERR_ZERO;
    } else {
        a = a1;
        if (!(PHT_BETA(0, a) > 0.0)) return PHT_UNIF_ERR_ZERO;
    }
    *B = a;

    /* 2. the visit states; x_j replaces beta_j(0), which no later draw reads */
    int prev = a;
    for (int j = 1; j <= m; j++) {
        const double gap = vt[j - 1] - (j > 1 ? vt[j - 2] : 0.0);
        const uint32_t mk = pht_unif_col_support(E, n, S, vo[j - 1]);
        int x;
        if (gap == 0.0) x = prev;
        else if ((mk & (mk - 1u)) == 0u) { x = 0; while (!((mk >> x) & 1u)) x++; }
        else {
            const double xx = lam * gap;
            pht_unif_exprow(tab, n, cap, xx, xx > 0.0 ? pht_log(xx) : 0.0, pht_unif_K(xx), prev, za, zs);
            for (int c = 0; c < n; c++) za[c * zs] = za[c * zs] * PHT_BETA(j, c);
            x = pht_unif_pick(za, n, zs, PHT_UNIF_U01(st));
            if (x < 0) return PHT_UNIF_ERR_ZERO;
        }
        PHT_BETA(j, 0) = (double)x;
        prev = x;
    }

    /* 3. the state at y */
    int b = prev;
    if (dy > 0.0) {
        const double xx = lam * dy;
        pht_unif_exprow(tab, n, cap, xx, xx > 0.0 ? pht_log(xx) : 0.0, pht_unif_K(xx), prev, za, zs);
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
        b = pht_unif_pick(za, n, zs, PHT_UNIF_U01(st));
        if (b < 0) return PHT_UNIF_ERR_ZERO;
    }
    for (int c = 0; c < n; c++) { za[c * zs] = 0.0; zb[c * zs] = 0.0; }

    /* 4. the bridges in time order */
    prev = a;
    for (int j = 1; j <= m + 1; j++) {
        const double gap = j > m ? dy : vt[j - 1] - (j > 1 ? vt[j - 2] : 0.0);
        const int x = j > m ? b : (int)PHT_BETA(j, 0);
        if (gap > 0.0) {
            const double xx = lam * gap;
            const int e = pht_unif_bridge(tab, n, cap, gap, xx, xx > 0.0 ? pht_log(xx) : 0.0, pht_unif_K(xx), prev, x, st, za, zb, zs, ctx);
            if (e) return e;
        }
        prev = x;
    }
#undef PHT_BETA

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
