// rm_math.h -- deterministic transcendental functions shared by the CUDA device code
// (NVRTC, sm_100a) and the host-side parity oracle (g++, -ffp-contract=off -mfma).
//
// Why this exists (SURVEY.md section 7, hard part H1): the reference's RNG is
//   gold_noise = fract(tan(distance(xy*PHI, xy)*seed)*xy.x)      raymarcher.frag:46-49
// which amplifies a 1-ULP change of tan() into a wholesale change of the sample.  GLSL ES 3.00
// leaves the precision of tan/sin/cos/log/pow/exp implementation-defined, so a parity
// check is only meaningful when kernel and oracle evaluate *the same* function.  Every
// function here is built exclusively from IEEE-754 binary64 operations that are correctly
// rounded on both x86-64 and sm_100 (add, mul, div, sqrt, fma, rint, int<->fp conversion,
// bit casts), with explicit fma() where fusion is wanted and no reliance on compiler
// contraction.  Identical source  =>  bit-identical float results on both sides.
//
// All functions take/return binary32 and evaluate in binary64; the results are within
// a fraction of an ULP of the correctly rounded value for arguments in the ranges GLSL
// code uses (|x| < 1e9 for the trigonometric family), deterministic everywhere else.
#ifndef RM_MATH_H_
#define RM_MATH_H_

// Under nvcc/NVRTC every function is __device__-only (the product has no host arithmetic);
// under g++ (the oracle) they are plain inline host functions.
#if defined(__CUDACC_RTC__) || defined(__CUDACC__)
#define RM_DEVICE_CODE 1
#define RM_HD __device__ __forceinline__
#else
#define RM_DEVICE_CODE 0
#define RM_HD inline
#include <cstring>
#include <cmath>
#endif

namespace rmx {

// ---------------------------------------------------------------- bit casts / primitives
// Bit casts go through memcpy on both sides (not the __double_as_longlong family): NVVM folds a
// memcpy bit cast at compile time, which lets calls with constant arguments - pow(uniform, i) in
// a specialised scene program - evaluate at compile time; the nvvm cast intrinsics do not fold.
#if RM_DEVICE_CODE
#define RM_MEMCPY memcpy
RM_HD double dfma(double a, double b, double c) { return fma(a, b, c); }
RM_HD double dfloor(double x) { return floor(x); }
RM_HD double dsqrt(double x) { return sqrt(x); }
#else
#define RM_MEMCPY __builtin_memcpy
RM_HD double dfma(double a, double b, double c) { return __builtin_fma(a, b, c); }
RM_HD double dfloor(double x) { return __builtin_floor(x); }
RM_HD double dsqrt(double x) { return __builtin_sqrt(x); }
#endif
RM_HD long long d2ll(double x) { long long r; RM_MEMCPY(&r, &x, 8); return r; }
RM_HD double ll2d(long long x) { double r; RM_MEMCPY(&r, &x, 8); return r; }
RM_HD int f2i(float x) { int r; RM_MEMCPY(&r, &x, 4); return r; }
RM_HD float i2f(int x) { float r; RM_MEMCPY(&r, &x, 4); return r; }
RM_HD double dabs(double x) { return ll2d(d2ll(x) & 0x7fffffffffffffffLL); }
// round to nearest even integer by the 2^52+2^51 trick: two IEEE additions, exact for
// |x| < 2^51, identity above (such doubles are already integers)
RM_HD double drint(double x) {
    const double M = 6755399441055744.0;
    if (!(dabs(x) < 2251799813685248.0)) return x;
    double t = x + M;
    return t - M;
}

RM_HD bool f_isnan(float x) { return (f2i(x) & 0x7fffffff) > 0x7f800000; }
RM_HD bool f_isinf(float x) { return (f2i(x) & 0x7fffffff) == 0x7f800000; }
RM_HD bool d_isnan(double x) { return (d2ll(x) & 0x7fffffffffffffffLL) > 0x7ff0000000000000LL; }
RM_HD float f_nan() { return i2f(0x7fffffff); }
RM_HD float f_inf() { return i2f(0x7f800000); }

// ---------------------------------------------------------------- trigonometric kernels
// Two sources for the same binary64 coefficients:
//   TrigLit  literals.  The compiler sees the values, so sin/cos/tan of compile-time constants (baked
//            uniforms in scene code) fold away; in generated code every 64-bit literal costs two UMOVs.
//   TrigTab  a table - on the device a (non-const) __constant__ array, which DFMA reads as
//            constant-bank operands (one LDCU.128 fetches two).  Used by the pipeline's RNG, where the
//            argument is never a constant and the literals were ~30 % of tan()'s instructions.
// Identical values, identical operations: results are bit-identical whichever source is used.
#define RM_TRIG_COEFFS                                                                                   \
    6.36619772367581382433e-01,  /*  0 2/pi */                                                           \
    1.57079632673412561417e+00,  /*  1 first 33 bits of pi/2 */                                          \
    6.07710050630396597660e-11,  /*  2 next 33 bits */                                                   \
    2.02226624879595063154e-21,  /*  3 remainder */                                                      \
    -1.66666666666666324348e-01, 8.33333333332248946124e-03, -1.98412698298579493134e-04, /* 4 S1..S6 */ \
    2.75573137070700676789e-06, -2.50507602534068634195e-08, 1.58969099521155010221e-10,                 \
    4.16666666666666019037e-02, -1.38888888888741095749e-03, 2.48015872894767294178e-05, /* 10 C1..C6 */ \
    -2.75573143513906633035e-07, 2.08757232129817482790e-09, -1.13596475577881948265e-11,                \
    6755399441055744.0,          /* 16 2^52 + 2^51 */                                                    \
    2147483648.0                 /* 17 2^31 */
#if RM_DEVICE_CODE
__device__ __constant__ double rm_trig_tab[18] = {RM_TRIG_COEFFS};
#else
static const double rm_trig_tab[18] = {RM_TRIG_COEFFS};
#endif
struct TrigTab { static RM_HD double at(int i) { return rm_trig_tab[i]; } };
struct TrigLit {
    static RM_HD double at(int i) {
        const double v[18] = {RM_TRIG_COEFFS};
        return v[i];
    }
};

// Reduction x = k*(pi/2) + r, |r| <= pi/4, three-term Cody-Waite with fma (constants are the
// classic split of pi/2 into 33-bit pieces).  k is returned modulo 4 in *quadrant.
template <class K>
RM_HD double trig_reduce(double x, int* quadrant) {
    const double xs = x * K::at(0);
    double k;
    if (dabs(xs) < K::at(17)) {
        // round-to-nearest-even by the 2^52+2^51 trick; the integer (two's complement) is then
        // sitting in the low mantissa bits of t, so k mod 4 is a mask - no floor / conversion
        const double t = xs + K::at(16);
        k = t - K::at(16);
        *quadrant = (int)(d2ll(t) & 3);
    } else {
        k = drint(xs);
        *quadrant = (int)dfma(-4.0, dfloor(k * 0.25), k);   // exact: k mod 4 in {0,1,2,3}
    }
    double r = dfma(-k, K::at(1), x);
    r = dfma(-k, K::at(2), r);
    r = dfma(-k, K::at(3), r);
    return r;
}

// sin(r), |r| <= pi/4  (odd minimax polynomial, degree 13)
template <class K>
RM_HD double ksin(double r) {
    double z = r * r;
    double p = dfma(z, K::at(9), K::at(8));
    p = dfma(z, p, K::at(7));
    p = dfma(z, p, K::at(6));
    p = dfma(z, p, K::at(5));
    p = dfma(z, p, K::at(4));
    return dfma(r * z, p, r);
}

// cos(r), |r| <= pi/4  (even minimax polynomial, degree 14)
template <class K>
RM_HD double kcos(double r) {
    double z = r * r;
    double p = dfma(z, K::at(15), K::at(14));
    p = dfma(z, p, K::at(13));
    p = dfma(z, p, K::at(12));
    p = dfma(z, p, K::at(11));
    p = dfma(z, p, K::at(10));
    return dfma(z * z, p, dfma(z, -0.5, 1.0));
}

template <class K>
RM_HD float sin_k(float x) {
    if (f_isnan(x) || f_isinf(x)) return f_nan();
    int q;
    double r = trig_reduce<K>((double)x, &q);
    double s = (q & 1) ? kcos<K>(r) : ksin<K>(r);
    if (q & 2) s = -s;
    if (x == 0.0f) return x;  // keep signed zero
    return (float)s;
}

template <class K>
RM_HD float cos_k(float x) {
    if (f_isnan(x) || f_isinf(x)) return f_nan();
    int q;
    double r = trig_reduce<K>((double)x, &q);
    double c = (q & 1) ? ksin<K>(r) : kcos<K>(r);
    if (((q + 1) & 2) != 0) c = -c;
    return (float)c;
}

template <class K>
RM_HD float tan_k(float x) {
    if (f_isnan(x) || f_isinf(x)) return f_nan();
    if (x == 0.0f) return x;
    int q;
    double r = trig_reduce<K>((double)x, &q);
    double s = ksin<K>(r), c = kcos<K>(r);
    // one division: -c/s in odd quadrants, s/c in even ones (operands selected first; same quotient bits)
    const double num = (q & 1) ? -c : s;
    const double den = (q & 1) ? s : c;
    return (float)(num / den);
}

// sin and cos of the same argument with one reduction and one pair of polynomials (Box-Muller);
// each result is bit-identical to sin_k / cos_k
template <class K>
RM_HD void sincos_k(float x, float* sn, float* cs) {
    if (f_isnan(x) || f_isinf(x)) { *sn = f_nan(); *cs = f_nan(); return; }
    int q;
    double r = trig_reduce<K>((double)x, &q);
    const double ps = ksin<K>(r), pc = kcos<K>(r);
    double s = (q & 1) ? pc : ps;
    if (q & 2) s = -s;
    double c = (q & 1) ? ps : pc;
    if (((q + 1) & 2) != 0) c = -c;
    *sn = (x == 0.0f) ? x : (float)s;
    *cs = (float)c;
}

// scene-code built-ins (foldable) and the pipeline's RNG versions (table-driven)
RM_HD float sin_f(float x) { return sin_k<TrigLit>(x); }
RM_HD float cos_f(float x) { return cos_k<TrigLit>(x); }
RM_HD float tan_f(float x) { return tan_k<TrigLit>(x); }
RM_HD float sin_ft(float x) { return sin_k<TrigTab>(x); }
RM_HD float cos_ft(float x) { return cos_k<TrigTab>(x); }
RM_HD float tan_ft(float x) { return tan_k<TrigTab>(x); }
RM_HD void sincos_ft(float x, float* sn, float* cs) { sincos_k<TrigTab>(x, sn, cs); }

// ---------------------------------------------------------------- log2 / exp2 in binary64
// Coefficients from literals (LeLit: foldable, scene code) or from a table (LeTab: pipeline code on
// the device, constant-bank operands) - see TrigLit / TrigTab above; same values, same results.
#define RM_LE_COEFFS                                                                                       \
    1.0 / 25.0, 1.0 / 23.0, 1.0 / 21.0, 1.0 / 19.0, 1.0 / 17.0, 1.0 / 15.0, 1.0 / 13.0, 1.0 / 11.0,      /*  0 atanh series */ \
    1.0 / 9.0, 1.0 / 7.0, 1.0 / 5.0, 1.0 / 3.0,                                                            \
    1.44269504088896338700e+00,                                                                /* 12 1/ln2 */ \
    1.41421356237309514547,                                                                    /* 13 sqrt2 */ \
    6.93147180559945286227e-01,                                                                /* 14 ln2   */ \
    1.0 / 87178291200.0, 1.0 / 6227020800.0, 1.0 / 479001600.0, 1.0 / 39916800.0, 1.0 / 3628800.0, /* 15 1/14! .. */ \
    1.0 / 362880.0, 1.0 / 40320.0, 1.0 / 5040.0, 1.0 / 720.0, 1.0 / 120.0, 1.0 / 24.0, 1.0 / 6.0     /* .. 26 1/3! */
#if RM_DEVICE_CODE
__device__ __constant__ double rm_le_tab[27] = {RM_LE_COEFFS};
#else
static const double rm_le_tab[27] = {RM_LE_COEFFS};
#endif
struct LeTab { static RM_HD double at(int i) { return rm_le_tab[i]; } };
struct LeLit {
    static RM_HD double at(int i) {
        const double v[27] = {RM_LE_COEFFS};
        return v[i];
    }
};

// log2(x) for finite x > 0 (denormal floats promoted to double are normal doubles).
template <class K>
RM_HD double dlog2_pos_k(double x) {
    long long b = d2ll(x);
    int e = (int)((b >> 52) & 0x7ff) - 1023;
    long long mb = (b & 0x000fffffffffffffLL) | 0x3ff0000000000000LL;
    double m = ll2d(mb);                                  // [1,2)
    if (m > K::at(13)) { m = m * 0.5; e += 1; }
    double f = m - 1.0;                                   // [-0.2929, 0.4142]
    double s = f / (2.0 + f);                             // |s| <= 0.1716
    double z = s * s;
    // atanh series: ln(m) = 2s(1 + z/3 + z^2/5 + ... ), 12 terms => < 1e-18 truncation
    double p = K::at(0);
    p = dfma(z, p, K::at(1));
    p = dfma(z, p, K::at(2));
    p = dfma(z, p, K::at(3));
    p = dfma(z, p, K::at(4));
    p = dfma(z, p, K::at(5));
    p = dfma(z, p, K::at(6));
    p = dfma(z, p, K::at(7));
    p = dfma(z, p, K::at(8));
    p = dfma(z, p, K::at(9));
    p = dfma(z, p, K::at(10));
    p = dfma(z, p, K::at(11));
    p = dfma(z, p, 1.0);
    double lnm = 2.0 * s * p;
    return dfma(lnm, K::at(12), (double)e);
}
RM_HD double dlog2_pos(double x) { return dlog2_pos_k<LeLit>(x); }

// 2^t for any double t; result is a double that converts to the wanted float
// (overflow -> +inf, underflow -> denormal/0 through the final conversion).
template <class K>
RM_HD double dexp2_k(double t) {
    if (d_isnan(t)) return t;
    if (t > 1000.0) t = 1000.0;
    if (t < -1000.0) t = -1000.0;
    double n = drint(t);
    double f = (t - n) * K::at(14);                       // f*ln2, |f| <= 0.3466
    // exp(f) Taylor to degree 14 (0.3466^15/15! ~ 1e-19)
    double p = K::at(15);
    p = dfma(f, p, K::at(16));
    p = dfma(f, p, K::at(17));
    p = dfma(f, p, K::at(18));
    p = dfma(f, p, K::at(19));
    p = dfma(f, p, K::at(20));
    p = dfma(f, p, K::at(21));
    p = dfma(f, p, K::at(22));
    p = dfma(f, p, K::at(23));
    p = dfma(f, p, K::at(24));
    p = dfma(f, p, K::at(25));
    p = dfma(f, p, K::at(26));
    p = dfma(f, p, 0.5);
    p = dfma(f, p, 1.0);
    p = dfma(f, p, 1.0);
    long long sb = ((long long)((int)n + 1023)) << 52;    // |n| <= 1000 so exponent is in range
    return p * ll2d(sb);
}
RM_HD double dexp2(double t) { return dexp2_k<LeLit>(t); }

// table-driven versions for pipeline code (RNG, shading, display): never constant arguments
RM_HD float log_ft(float x) {
    if (f_isnan(x) || x < 0.0f) return f_nan();
    if (x == 0.0f) return -f_inf();
    if (f_isinf(x)) return x;
    return (float)(dlog2_pos_k<LeTab>((double)x) * LeTab::at(14));
}
RM_HD float exp_ft(float x) { return (float)dexp2_k<LeTab>((double)x * LeTab::at(12)); }

RM_HD float log2_f(float x) {
    if (f_isnan(x) || x < 0.0f) return f_nan();
    if (x == 0.0f) return -f_inf();
    if (f_isinf(x)) return x;
    return (float)dlog2_pos((double)x);
}

RM_HD float log_f(float x) {
    if (f_isnan(x) || x < 0.0f) return f_nan();
    if (x == 0.0f) return -f_inf();
    if (f_isinf(x)) return x;
    return (float)(dlog2_pos((double)x) * 6.93147180559945286227e-01);
}

// ---------------------------------------------------------------- fast paths of the pipeline's RNG functions
// tan_ft, sincos_ft and log_ft end in a conversion to float: their binary64 value P only has to pick (float)P.
// For the arguments the RNG produces, each fast path below computes a cheaper binary64 value F - no special-case
// branches, no correctly rounded division - with |F - P| <= D units in the last place of F, and returns (float)F
// only when F is farther than D ulps from every float rounding boundary (the midpoint between two floats, where
// the 29 mantissa bits a float drops read 2^28).  Every value within D ulps of F then rounds to the same float as
// F, so the result equals the pinned function's by construction.  A binade edge is no rounding boundary, and the
// nearest boundary across one is 2^24 ulps away, so F and P in neighbouring binades need no special case.  Near a
// boundary, and outside the domain, the pinned function runs, out of line.  In the tan and log domains every
// result is a normal float or zero, so F's binade sets the rounding boundaries.  Only IEEE binary64 operations are used (dmul / dadd where an unfused result is meant, whatever
// --fmad says), so a host build computes the same F: tools/rng_sweep.py checks every float of each domain and
// measures the largest |F - P|, which D exceeds at least fourfold.
#if RM_DEVICE_CODE
#define RM_COLD __device__ __noinline__
RM_HD double dmul(double a, double b) { return __dmul_rn(a, b); }
RM_HD double dadd(double a, double b) { return __dadd_rn(a, b); }
#else
#define RM_COLD inline
RM_HD double dmul(double a, double b) { return a * b; }
RM_HD double dadd(double a, double b) { return a + b; }
#endif
struct SinCos { float s, c; };
RM_COLD float tan_ft_pinned(float x) { return tan_ft(x); }
RM_COLD SinCos sincos_ft_pinned(float x) { SinCos r; sincos_ft(x, &r.s, &r.c); return r; }
RM_COLD float log_ft_pinned(float x) { return log_ft(x); }

// F is farther than D ulps (of F) from every float rounding boundary
RM_HD bool rounds_clear(double F, unsigned D) {
    const unsigned low = (unsigned)d2ll(F) & 0x1fffffffu;
    return low - (0x10000000u - D) > 2u * D;
}
// n / a for a > 0 normal, within 1 ulp: a bit-pattern estimate of 1/a (relative error < 0.051), three Newton steps
// (< 2^-34), then one correction of the quotient (error ~ 2^-68 plus its rounding)
RM_HD double div_pos(double n, double a) {
    double y = ll2d(0x7FDE623822FC16E6LL - d2ll(a));
    double e = dfma(-a, y, 1.0);
    y = dfma(y, e, y);
    e = dfma(-a, y, 1.0);
    y = dfma(y, e, y);
    e = dfma(-a, y, 1.0);
    y = dfma(y, e, y);
    const double q = dmul(n, y);
    return dfma(dfma(-a, q, n), y, q);
}

// tan_ft on [2^-126, 1024): the pinned reduction (here |x * 2/pi| < 2^31 always takes its first path), then
// tan r = r + r z P(z) / Q(z), z = r^2, the rational approximation of the Cephes library's tan.c (S. L. Moshier;
// relative error ~2^-52 on |r| <= pi/4) in place of two polynomials, and the quotient by div_pos.  P and Q are
// stored negated, so Q > 0.
#define RM_TAN_FAST_COEFFS                                                                            \
    1.30936939181383777646e+04, -1.15351664838587416140e+06, 1.79565251976484877988e+07, /* 0 -P */ \
    -1.36812963470692954678e+04, 1.32089234440210967447e+06, -2.50083801823357915839e+07,            \
    5.38695755929454629881e+07                                                           /* 3 -Q */
#if RM_DEVICE_CODE
__device__ __constant__ double rm_tan_tab[7] = {RM_TAN_FAST_COEFFS};
#else
static const double rm_tan_tab[7] = {RM_TAN_FAST_COEFFS};
#endif
constexpr unsigned RM_TAN_FAST_D = 16;
RM_HD double tan_ft_fast_value(float x) {
    typedef TrigTab K;
    const double xd = (double)x;
    const double t = dadd(dmul(xd, K::at(0)), K::at(16));
    const double k = dadd(t, -K::at(16));
    double r = dfma(-k, K::at(1), xd);
    r = dfma(-k, K::at(2), r);
    r = dfma(-k, K::at(3), r);
    const double z = dmul(r, r);
    double p = dfma(z, rm_tan_tab[0], rm_tan_tab[1]);
    p = dfma(z, p, rm_tan_tab[2]);
    double q = dadd(-z, rm_tan_tab[3]);
    q = dfma(z, q, rm_tan_tab[4]);
    q = dfma(z, q, rm_tan_tab[5]);
    q = dfma(z, q, rm_tan_tab[6]);
    const double n = dfma(dmul(r, z), p, dmul(r, q));       // tan r = n / q, n has the sign of r
    // n / q in even quadrants; -q / n in odd ones, as q / -n so that the divisor is positive
    const bool odd = (d2ll(t) & 1) != 0;
    const double num = odd ? (r < 0.0 ? q : -q) : n;
    const double den = odd ? dabs(n) : q;
    return div_pos(num, den);
}
RM_HD float tan_ft_fast(float x) {
    if ((unsigned)(f2i(x) - 0x00800000) >= (unsigned)(0x44800000 - 0x00800000)) return tan_ft_pinned(x);
    const double F = tan_ft_fast_value(x);
    if (!rounds_clear(F, RM_TAN_FAST_D)) return tan_ft_pinned(x);
    return (float)F;
}

// sincos_ft on [+0, 8): the pinned operations without the special cases and the second reduction path, so F == P
// and no rounding test is needed
RM_HD void sincos_ft_fast(float x, float* sn, float* cs) {
    if ((unsigned)f2i(x) >= 0x41000000u) {
        const SinCos p = sincos_ft_pinned(x);
        *sn = p.s;
        *cs = p.c;
        return;
    }
    typedef TrigTab K;
    const double xd = (double)x;
    const double t = dadd(dmul(xd, K::at(0)), K::at(16));
    const double k = dadd(t, -K::at(16));
    const int q = (int)(d2ll(t) & 3);
    double r = dfma(-k, K::at(1), xd);
    r = dfma(-k, K::at(2), r);
    r = dfma(-k, K::at(3), r);
    const double ps = ksin<K>(r), pc = kcos<K>(r);
    double s = (q & 1) ? pc : ps;
    if (q & 2) s = -s;
    double c = (q & 1) ? ps : pc;
    if (((q + 1) & 2) != 0) c = -c;
    *sn = (float)s;
    *cs = (float)c;
}

// log_ft on [2^-126, 1]: the pinned mantissa split, s = f / (2 + f) by div_pos, the atanh series to z^9 (the
// omitted terms are below 2^-50 of the sum), and ln x = e ln2 + ln m in one fma
constexpr unsigned RM_LOG_FAST_D = 8;
RM_HD double log_ft_fast_value(float x) {
    typedef LeTab K;
    const long long b = d2ll((double)x);
    int e = (int)(b >> 52) - 1023;
    double m = ll2d((b & 0x000fffffffffffffLL) | 0x3ff0000000000000LL);
    if (m > K::at(13)) { m = dmul(m, 0.5); e += 1; }
    const double f = dadd(m, -1.0);
    const double s = div_pos(f, dadd(2.0, f));
    const double z = dmul(s, s);
    double p = K::at(3);
    p = dfma(z, p, K::at(4));
    p = dfma(z, p, K::at(5));
    p = dfma(z, p, K::at(6));
    p = dfma(z, p, K::at(7));
    p = dfma(z, p, K::at(8));
    p = dfma(z, p, K::at(9));
    p = dfma(z, p, K::at(10));
    p = dfma(z, p, K::at(11));
    p = dfma(z, p, 1.0);
    return dfma((double)e, K::at(14), dmul(dadd(s, s), p));
}
RM_HD float log_ft_fast(float x) {
    if ((unsigned)(f2i(x) - 0x00800000) > (unsigned)(0x3f800000 - 0x00800000)) return log_ft_pinned(x);
    const double F = log_ft_fast_value(x);
    if (!rounds_clear(F, RM_LOG_FAST_D)) return log_ft_pinned(x);
    return (float)F;
}

RM_HD float exp2_f(float x) { return (float)dexp2((double)x); }

RM_HD float exp_f(float x) { return (float)dexp2((double)x * 1.44269504088896338700e+00); }

// pow(x, y).  GLSL ES 3.00 leaves x < 0 undefined; the reference relies on pow(negative, 2.0)
// being a square (schlick(), raymarcher.frag:173, with n1 < n2), which is what GPU compilers
// deliver by strength-reducing constant integer exponents.  Pinned: C99 powf semantics - a
// negative base with an integral exponent gives +-|x|^y, otherwise NaN; pow(x,0)=1, pow(0,y>0)=0.
template <class K>
RM_HD float pow_k(float x, float y) {
    if (f_isnan(x) || f_isnan(y)) return f_nan();
    if (y == 0.0f) return 1.0f;
    bool negate = false;
    if (x < 0.0f) {
        double yd = (double)y;
        if (f_isinf(y)) { x = -x; }
        else {
            if (yd != drint(yd)) return f_nan();
            double h = yd * 0.5;
            negate = (h != drint(h)) && (dabs(yd) < 16777216.0);   // odd integer exponent
            x = -x;
        }
    }
    float r;
    if (x == 0.0f) r = (y > 0.0f) ? 0.0f : f_inf();
    else if (f_isinf(x)) r = (y > 0.0f) ? f_inf() : 0.0f;
    else if (x == 1.0f) r = 1.0f;
    else if (f_isinf(y)) {
        bool grow = (x > 1.0f) == (y > 0.0f);
        r = grow ? f_inf() : 0.0f;
    } else r = (float)dexp2_k<K>((double)y * dlog2_pos_k<K>((double)x));
    return negate ? -r : r;
}
RM_HD float pow_f(float x, float y) { return pow_k<LeLit>(x, y); }
RM_HD float pow_ft(float x, float y) { return pow_k<LeTab>(x, y); }

// ---------------------------------------------------------------- inverse trigonometric
// atan for a double argument, result in (-pi/2, pi/2).
RM_HD double datan(double x) {
    const double PIO2 = 1.57079632679489655800e+00;
    bool neg = x < 0.0;
    double a = neg ? -x : x;
    bool inv = a > 1.0;
    if (inv) a = 1.0 / a;
    // two argument halvings: atan(a) = 2 atan(a / (1 + sqrt(1 + a^2)))  -> |a| <= 0.1990
    a = a / (1.0 + dsqrt(dfma(a, a, 1.0)));
    a = a / (1.0 + dsqrt(dfma(a, a, 1.0)));
    double z = a * a;
    double p = -1.0 / 23.0;
    p = dfma(z, p, 1.0 / 21.0);
    p = dfma(z, p, -1.0 / 19.0);
    p = dfma(z, p, 1.0 / 17.0);
    p = dfma(z, p, -1.0 / 15.0);
    p = dfma(z, p, 1.0 / 13.0);
    p = dfma(z, p, -1.0 / 11.0);
    p = dfma(z, p, 1.0 / 9.0);
    p = dfma(z, p, -1.0 / 7.0);
    p = dfma(z, p, 1.0 / 5.0);
    p = dfma(z, p, -1.0 / 3.0);
    p = dfma(z, p, 1.0);
    double r = 4.0 * a * p;
    if (inv) r = PIO2 - r;
    return neg ? -r : r;
}

RM_HD double datan2(double y, double x) {
    const double PI = 3.14159265358979311600e+00;
    const double PIO2 = 1.57079632679489655800e+00;
    if (d_isnan(x) || d_isnan(y)) return x + y;
    if (x == 0.0) {
        if (y == 0.0) return 0.0;
        return y > 0.0 ? PIO2 : -PIO2;
    }
    double ax = dabs(x), ay = dabs(y);
    double r;
    if (ax >= ay) r = datan(ay / ax); else r = PIO2 - datan(ax / ay);
    if (x < 0.0) r = PI - r;
    return y < 0.0 ? -r : r;
}

RM_HD float atan_f(float x) {
    if (f_isnan(x)) return f_nan();
    if (f_isinf(x)) return x > 0.0f ? 1.57079637f : -1.57079637f;
    if (x == 0.0f) return x;
    return (float)datan((double)x);
}
RM_HD float atan2_f(float y, float x) {
    if (f_isnan(x) || f_isnan(y)) return f_nan();
    if (f_isinf(x) || f_isinf(y)) {
        // map infinities to unit steps: (inf,inf) -> 45 degree family, one-sided -> axis
        double dx = f_isinf(x) ? (x > 0.0f ? 1.0 : -1.0) : 0.0;
        double dy = f_isinf(y) ? (y > 0.0f ? 1.0 : -1.0) : 0.0;
        if (dy == 0.0) {
            double r = dx > 0.0 ? 0.0 : 3.14159265358979311600e+00;
            return (float)(y < 0.0f ? -r : r);
        }
        return (float)datan2(dy, dx);
    }
    return (float)datan2((double)y, (double)x);
}
RM_HD float asin_f(float x) {
    if (f_isnan(x) || x > 1.0f || x < -1.0f) return f_nan();
    if (x == 0.0f) return x;
    double d = (double)x;
    return (float)datan2(d, dsqrt((1.0 - d) * (1.0 + d)));
}
RM_HD float acos_f(float x) {
    if (f_isnan(x) || x > 1.0f || x < -1.0f) return f_nan();
    double d = (double)x;
    return (float)datan2(dsqrt((1.0 - d) * (1.0 + d)), d);
}

// ---------------------------------------------------------------- hyperbolic family
RM_HD double dexp(double x) { return dexp2(x * 1.44269504088896338700e+00); }
RM_HD double dlog(double x) { return dlog2_pos(x) * 6.93147180559945286227e-01; }

RM_HD float sinh_f(float x) {
    if (f_isnan(x)) return f_nan();
    if (x == 0.0f || f_isinf(x)) return x;
    double d = (double)x;
    if (dabs(d) < 1e-4) return (float)dfma(d * d * d, 1.0 / 6.0, d);
    if (dabs(d) > 700.0) return d > 0.0 ? f_inf() : -f_inf();
    double e = dexp(d);
    return (float)(0.5 * (e - 1.0 / e));
}
RM_HD float cosh_f(float x) {
    if (f_isnan(x)) return f_nan();
    if (f_isinf(x)) return f_inf();
    double d = dabs((double)x);
    if (d > 700.0) return f_inf();
    double e = dexp(d);
    return (float)(0.5 * (e + 1.0 / e));
}
RM_HD float tanh_f(float x) {
    if (f_isnan(x)) return f_nan();
    if (x == 0.0f) return x;
    double d = (double)x;
    if (dabs(d) > 20.0) return d > 0.0 ? 1.0f : -1.0f;
    if (dabs(d) < 1e-4) return (float)dfma(d * d * d, -1.0 / 3.0, d);
    double e = dexp(2.0 * d);
    return (float)((e - 1.0) / (e + 1.0));
}
RM_HD float asinh_f(float x) {
    if (f_isnan(x)) return f_nan();
    if (x == 0.0f || f_isinf(x)) return x;
    double d = dabs((double)x);
    double r = (d < 1e-4) ? dfma(d * d * d, -1.0 / 6.0, d) : dlog(d + dsqrt(dfma(d, d, 1.0)));
    return (float)(x < 0.0f ? -r : r);
}
RM_HD float acosh_f(float x) {
    if (f_isnan(x) || x < 1.0f) return f_nan();
    if (f_isinf(x)) return x;
    double d = (double)x;
    return (float)dlog(d + dsqrt((d - 1.0) * (d + 1.0)));
}
RM_HD float atanh_f(float x) {
    if (f_isnan(x) || x > 1.0f || x < -1.0f) return f_nan();
    if (x == 0.0f) return x;
    if (x == 1.0f) return f_inf();
    if (x == -1.0f) return -f_inf();
    double d = (double)x;
    if (dabs(d) < 1e-4) return (float)dfma(d * d * d, 1.0 / 3.0, d);
    return (float)(0.5 * dlog((1.0 + d) / (1.0 - d)));
}

}  // namespace rmx

#endif  // RM_MATH_H_
