/*
 * pht_math.h -- bit-reproducible FP64 exp/log shared by the CUDA kernels and
 * the host-side checkers.
 *
 * Why this exists: tier-1 parity (BASELINE.json north_star) asks for bit-exact
 * integer sufficient statistics against the reference C samplers.  Every
 * categorical scan, ARMS accept/squeeze test and Brent branch in the reference
 * (e.g. src/Simulate_AbsCTMC_gt_Bladt_MHRS.c:61,101; src/arms.c:464;
 * src/utility.c:273-331) is a floating-point comparison, so a 1-ulp difference
 * between glibc's and CUDA's libm flips decisions.  Both sides therefore use
 * THIS implementation: the device code calls pht_exp/pht_log directly and the
 * reference build links `exp`/`log` to them (oracle/shim/rshim.c).  Only
 * IEEE-754 add/mul/div and explicitly written fma() are used, evaluated in a
 * fixed order; host code must be built with -ffp-contract=off and device code
 * with -fmad=false so neither compiler introduces contractions of its own.
 *
 * Accuracy: < 1 ulp for both functions (checked against libm in
 * tests/test_math.py).  Algorithms are the classical ones: Cody-Waite range
 * reduction + Taylor/Horner for exp, the fdlibm-style atanh series for log.
 */
#ifndef PHT_MATH_H
#define PHT_MATH_H

#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define PHT_HD __host__ __device__ __forceinline__
#else
#define PHT_HD static inline
#endif

#if defined(__CUDA_ARCH__)
#define PHT_FMA(a, b, c) __fma_rn((a), (b), (c))
#else
#define PHT_FMA(a, b, c) __builtin_fma((a), (b), (c))
#endif

PHT_HD uint64_t pht_d2u(double x) {
#if defined(__CUDA_ARCH__)
    return (uint64_t)__double_as_longlong(x);
#else
    uint64_t u; memcpy(&u, &x, 8); return u;
#endif
}
PHT_HD double pht_u2d(uint64_t u) {
#if defined(__CUDA_ARCH__)
    return __longlong_as_double((long long)u);
#else
    double x; memcpy(&x, &u, 8); return x;
#endif
}

/* Polynomial coefficients.  On the device they live in constant memory so that each one is an operand of its
 * FMA (a 64-bit literal would cost two moves per use); the host uses the same values as literals. */
#define PHT_EXP_COEFFS \
    1.6059043836821613e-10, 2.08767569878681e-09, 2.505210838544172e-08, 2.755731922398589e-07, \
    2.7557319223985893e-06, 2.48015873015873e-05, 1.984126984126984e-04, 1.388888888888889e-03, \
    8.333333333333333e-03, 4.1666666666666664e-02, 1.6666666666666666e-01, 0.5, 1.0, 1.0      /* 1/13! ... 1/2!, 1, 1 */
#define PHT_LOG_COEFFS \
    6.666666666666735130e-01, 3.999999999940941908e-01, 2.857142874366239149e-01, 2.222219843214978396e-01, \
    1.818357216161805012e-01, 1.531383769920937332e-01, 1.479819860511658591e-01                  /* L1 ... L7 (fdlibm e_log.c) */
#if defined(__CUDACC__)
static __constant__ double pht_exp_cd[14] = { PHT_EXP_COEFFS };
static __constant__ double pht_log_cd[7] = { PHT_LOG_COEFFS };
#endif
static const double pht_exp_ch[14] = { PHT_EXP_COEFFS };
static const double pht_log_ch[7] = { PHT_LOG_COEFFS };
#if defined(__CUDA_ARCH__)
#define PHT_EC(i) pht_exp_cd[i]
#define PHT_LC(i) pht_log_cd[i]
#define PHT_SLOW __device__ __noinline__
#else
#define PHT_EC(i) pht_exp_ch[i]
#define PHT_LC(i) pht_log_ch[i]
#define PHT_SLOW static
#endif

/* exp(x).  k = round(x/ln2); r = x - k ln2 (two-step, fma); Taylor degree 13 on |r| <= ln2/2 (remainder < 5e-18
 * relative); result p * 2^k.
 * Fast path |x| <= 708: p is in [0.70, 1.42] and |k| <= 1021, so p * 2^k is a normal number and the scaling is
 * exact: it is done by adding k to the exponent field.  Everything else (NaN, overflow, results near or below
 * the subnormal range) takes the general path, which scales in two exact halves.  Both paths compute the same
 * value wherever both apply, so the split is invisible in the results. */
PHT_SLOW double pht_exp_general(double x) {
    if (!(x == x)) return x + x;                          /* NaN */
    if (x > 709.782712893384) return pht_u2d(0x7ff0000000000000ULL);
    if (x < -745.1332191019412) return 0.0;
    const double LOG2E  = 1.4426950408889634074;          /* 1/ln2 */
    const double LN2_HI = 6.93147180559945286227e-01;     /* nearest double to ln2 */
    const double LN2_LO = 2.31904681384629955842e-17;     /* ln2 - LN2_HI */
    const double SHIFT  = 6755399441055744.0;             /* 1.5 * 2^52 */
    double kd = PHT_FMA(x, LOG2E, SHIFT) - SHIFT;          /* round-to-nearest integer */
    double r = PHT_FMA(-kd, LN2_HI, x);
    r = PHT_FMA(-kd, LN2_LO, r);
    double p = PHT_EC(0);
    for (int i = 1; i < 14; i++) p = PHT_FMA(p, r, PHT_EC(i));
    int k = (int)kd;
    int k1 = k >> 1, k2 = k - k1;                         /* both within [-538, 512] */
    double s1 = pht_u2d((uint64_t)(int64_t)(k1 + 1023) << 52);
    double s2 = pht_u2d((uint64_t)(int64_t)(k2 + 1023) << 52);
    return (p * s1) * s2;
}

PHT_HD double pht_exp(double x) {
    const double LOG2E  = 1.4426950408889634074;
    const double LN2_HI = 6.93147180559945286227e-01;
    const double LN2_LO = 2.31904681384629955842e-17;
    const double SHIFT  = 6755399441055744.0;
    if (!(__builtin_fabs(x) <= 708.0)) return pht_exp_general(x);
    const double t = PHT_FMA(x, LOG2E, SHIFT);
    const double kd = t - SHIFT;
    double r = PHT_FMA(-kd, LN2_HI, x);
    r = PHT_FMA(-kd, LN2_LO, r);
    double p = PHT_EC(0);
    p = PHT_FMA(p, r, PHT_EC(1));  p = PHT_FMA(p, r, PHT_EC(2));  p = PHT_FMA(p, r, PHT_EC(3));
    p = PHT_FMA(p, r, PHT_EC(4));  p = PHT_FMA(p, r, PHT_EC(5));  p = PHT_FMA(p, r, PHT_EC(6));
    p = PHT_FMA(p, r, PHT_EC(7));  p = PHT_FMA(p, r, PHT_EC(8));  p = PHT_FMA(p, r, PHT_EC(9));
    p = PHT_FMA(p, r, PHT_EC(10)); p = PHT_FMA(p, r, PHT_EC(11)); p = PHT_FMA(p, r, PHT_EC(12));
    p = PHT_FMA(p, r, PHT_EC(13));
    /* the low mantissa word of t = k + 1.5 * 2^52 holds k in two's complement */
#if defined(__CUDA_ARCH__)
    const int k = __double2loint(t);
    return __hiloint2double(__double2hiint(p) + (k << 20), __double2loint(p));
#else
    const int k = (int)(uint32_t)pht_d2u(t);
    return pht_u2d(pht_d2u(p) + ((uint64_t)(int64_t)k << 52));
#endif
}

#if defined(__CUDACC__)
/* Four exponentials side by side: the same operations per element as pht_exp (so the same bits), with the four dependent
 * chains (3 + 13 FMAs of ~8 cycles each) interleaved -- the kernels that evaluate spectral sums run 4-5 warps per
 * scheduler and were waiting on exactly these chains.  Falls back to pht_exp when an argument is outside the fast range. */
static __device__ __forceinline__ void pht_exp4(const double x0, const double x1, const double x2, const double x3,
                                                double &e0, double &e1, double &e2, double &e3) {
    const double LOG2E  = 1.4426950408889634074;
    const double LN2_HI = 6.93147180559945286227e-01;
    const double LN2_LO = 2.31904681384629955842e-17;
    const double SHIFT  = 6755399441055744.0;
    const bool ok = (__builtin_fabs(x0) <= 708.0) && (__builtin_fabs(x1) <= 708.0) && (__builtin_fabs(x2) <= 708.0) && (__builtin_fabs(x3) <= 708.0);
    if (!ok) { e0 = pht_exp(x0); e1 = pht_exp(x1); e2 = pht_exp(x2); e3 = pht_exp(x3); return; }
    const double t0 = PHT_FMA(x0, LOG2E, SHIFT), t1 = PHT_FMA(x1, LOG2E, SHIFT), t2 = PHT_FMA(x2, LOG2E, SHIFT), t3 = PHT_FMA(x3, LOG2E, SHIFT);
    const double k0 = t0 - SHIFT, k1 = t1 - SHIFT, k2 = t2 - SHIFT, k3 = t3 - SHIFT;
    double r0 = PHT_FMA(-k0, LN2_HI, x0), r1 = PHT_FMA(-k1, LN2_HI, x1), r2 = PHT_FMA(-k2, LN2_HI, x2), r3 = PHT_FMA(-k3, LN2_HI, x3);
    r0 = PHT_FMA(-k0, LN2_LO, r0); r1 = PHT_FMA(-k1, LN2_LO, r1); r2 = PHT_FMA(-k2, LN2_LO, r2); r3 = PHT_FMA(-k3, LN2_LO, r3);
    double p0 = PHT_EC(0), p1 = PHT_EC(0), p2 = PHT_EC(0), p3 = PHT_EC(0);
#define PHT_E4(c) p0 = PHT_FMA(p0, r0, PHT_EC(c)); p1 = PHT_FMA(p1, r1, PHT_EC(c)); p2 = PHT_FMA(p2, r2, PHT_EC(c)); p3 = PHT_FMA(p3, r3, PHT_EC(c));
    PHT_E4(1) PHT_E4(2) PHT_E4(3) PHT_E4(4) PHT_E4(5) PHT_E4(6) PHT_E4(7) PHT_E4(8) PHT_E4(9) PHT_E4(10) PHT_E4(11) PHT_E4(12) PHT_E4(13)
#undef PHT_E4
    e0 = __hiloint2double(__double2hiint(p0) + (__double2loint(t0) << 20), __double2loint(p0));
    e1 = __hiloint2double(__double2hiint(p1) + (__double2loint(t1) << 20), __double2loint(p1));
    e2 = __hiloint2double(__double2hiint(p2) + (__double2loint(t2) << 20), __double2loint(p2));
    e3 = __hiloint2double(__double2hiint(p3) + (__double2loint(t3) << 20), __double2loint(p3));
}
#endif

/* log(x).  x = 2^e * m, m in [sqrt(1/2), sqrt(2)); f = m - 1; s = f/(2+f);
 * log(1+f) = f - f^2/2 + s*(f^2/2 + R(s^2)) with the degree-7 even polynomial
 * R from fdlibm (e_log.c; Sun Microsystems 1993, freely distributable).
 * pht_log_core is the computation for a positive normal x; pht_log adds the special cases. */
PHT_HD double pht_log_core(uint64_t ux, int e) {
    const double LN2_HI = 6.93147180369123816490e-01;     /* 0x3fe62e42fee00000 */
    const double LN2_LO = 1.90821492927058770002e-10;     /* 0x3dea39ef35793c76 */
    /* bring the mantissa into [sqrt(1/2), sqrt(2)) */
    uint32_t hx = (uint32_t)(ux >> 32);
    hx += 0x3ff00000u - 0x3fe6a09eu;
    e += (int)(hx >> 20) - 0x3ff;
    hx = (hx & 0x000fffffu) + 0x3fe6a09eu;
    double m = pht_u2d(((uint64_t)hx << 32) | (ux & 0xffffffffULL));
    double f = m - 1.0;
    double hfsq = 0.5 * f * f;
    double s = f / (2.0 + f);
    double z = s * s;
    double w = z * z;
    double t1 = w * PHT_FMA(w, PHT_FMA(w, PHT_LC(5), PHT_LC(3)), PHT_LC(1));
    double t2 = z * PHT_FMA(w, PHT_FMA(w, PHT_FMA(w, PHT_LC(6), PHT_LC(4)), PHT_LC(2)), PHT_LC(0));
    double R = t2 + t1;
    double dk = (double)e;
    return dk * LN2_HI - ((hfsq - (s * (hfsq + R) + dk * LN2_LO)) - f);
}

PHT_SLOW double pht_log_special(double x) {
    uint64_t ux = pht_d2u(x);
    if (ux >= 0x7ff0000000000000ULL) {                    /* inf, NaN, negative */
        if (ux == 0x7ff0000000000000ULL) return x;        /* +inf */
        if (!(x == x)) return x + x;                      /* NaN */
        if (x == 0.0) return -pht_u2d(0x7ff0000000000000ULL);   /* -0 */
        return pht_u2d(0x7ff8000000000000ULL);            /* x < 0 */
    }
    if (ux == 0) return -pht_u2d(0x7ff0000000000000ULL);  /* +0 */
    x *= 18014398509481984.0;                             /* subnormal: scale by 2^54 */
    return pht_log_core(pht_d2u(x), -54);
}

PHT_HD double pht_log(double x) {
    const uint64_t ux = pht_d2u(x);
    if (ux - 0x0010000000000000ULL >= 0x7fe0000000000000ULL) return pht_log_special(x);   /* not a positive normal */
    return pht_log_core(ux, 0);
}

/* log(1 + x), fdlibm's s_log1p.c on the polynomial of pht_log (its Lp1..Lp7 are the Lg1..Lg7 above).
 * Fast path: 1 + x in [sqrt(1/2), sqrt(2)), i.e. x in [-0.2929, 0.4142): f = x exactly and no reduction.  The general
 * path takes every x: on the fast range it computes what the fast path computes; elsewhere it reduces u = 1 + x to
 * 2^k m like pht_log and carries the rounding of u as the correction c = (x - (u - 1)) / u (also where the reduction
 * gives k = 0, at the edges of the fast range, which fdlibm drops). */
#define PHT_LOG1P_LO (-0.2928932188134524)        /* sqrt(1/2) - 1 */
#define PHT_LOG1P_HI 0.41421356237309503          /* sqrt(2) - 1 */
PHT_HD double pht_log1p_poly(double f, double *hfsq, double *s) {
    *hfsq = 0.5 * f * f;
    *s = f / (2.0 + f);
    const double z = *s * *s;
    const double w = z * z;
    const double t1 = w * PHT_FMA(w, PHT_FMA(w, PHT_LC(5), PHT_LC(3)), PHT_LC(1));
    const double t2 = z * PHT_FMA(w, PHT_FMA(w, PHT_FMA(w, PHT_LC(6), PHT_LC(4)), PHT_LC(2)), PHT_LC(0));
    return t2 + t1;
}
PHT_SLOW double pht_log1p_general(double x) {
    if (!(x == x)) return x + x;                                  /* NaN */
    if (x < -1.0) return pht_u2d(0x7ff8000000000000ULL);
    if (x == -1.0) return -pht_u2d(0x7ff0000000000000ULL);
    if (x == pht_u2d(0x7ff0000000000000ULL)) return x;
    const double LN2_HI = 6.93147180369123816490e-01;
    const double LN2_LO = 1.90821492927058770002e-10;
    double hfsq, s;
    if (x >= PHT_LOG1P_LO && x < PHT_LOG1P_HI) {
        const double R = pht_log1p_poly(x, &hfsq, &s);
        return x - (hfsq - s * (hfsq + R));
    }
    const double u = x < 9007199254740992.0 ? 1.0 + x : x;         /* beyond 2^53, 1 + x rounds to x: no correction */
    const uint64_t uu = pht_d2u(u);
    uint32_t hu = (uint32_t)(uu >> 32);
    int k = (int)(hu >> 20) - 1023;
    const double c = x < 9007199254740992.0 ? (k > 0 ? 1.0 - (u - x) : x - (u - 1.0)) / u : 0.0;
    hu &= 0x000fffffu;
    if (hu < 0x6a09eu) hu |= 0x3ff00000u;                          /* mantissa in [1, sqrt(2)) */
    else { k += 1; hu |= 0x3fe00000u; }                              /* in [sqrt(1/2), 1) */
    const double f = pht_u2d(((uint64_t)hu << 32) | (uu & 0xffffffffULL)) - 1.0;
    const double R = pht_log1p_poly(f, &hfsq, &s);
    const double dk = (double)k;
    return dk * LN2_HI - ((hfsq - (s * (hfsq + R) + (dk * LN2_LO + c))) - f);
}
PHT_HD double pht_log1p(double x) {
    if (!(x >= PHT_LOG1P_LO && x < PHT_LOG1P_HI)) return pht_log1p_general(x);
    double hfsq, s;
    const double R = pht_log1p_poly(x, &hfsq, &s);
    return x - (hfsq - s * (hfsq + R));
}

#endif /* PHT_MATH_H */
