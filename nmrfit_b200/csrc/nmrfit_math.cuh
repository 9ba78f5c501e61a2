// Device math for the Voigt / Kramers-Kronig lineshapes (sm_100a).
//
// Everything the inner loops evaluate lives here so that it can also be compiled
// for the host (tests/host_math_harness.cpp defines NMRFIT_HOST_MATH and empties
// the CUDA qualifiers) and checked against libm/mpmath without a GPU.  The host
// build exists only for those accuracy tests; the product never runs it.
//
// Cost accounting (FP64-pipe issue slots; DFMA/DMUL/DADD = 1 slot each):
//   rcp_pos      3 slots + 1 MUFU.RCP64H
//   exp_neg<0>   15 slots   (degree-11 polynomial, no table)
//   exp_neg<6>    9 slots   (64-entry 2^(j/64) table in shared memory, degree 5)
//   exp_neg<8>    8 slots   (256-entry table, degree 4)
//   exp_neg<10>   7 slots   (1024-entry table, degree 3)
#pragma once
#include "nmrfit_coeffs.cuh"
#include "objective_smem.h"     // kFarPoly

#ifdef NMRFIT_HOST_MATH
#include <cmath>
#include <cstring>
#include <cstdint>
#define NMRFIT_HD inline
static inline int nmrfit_hi(double x) { int64_t b; std::memcpy(&b, &x, 8); return (int)(b >> 32); }
static inline int nmrfit_lo(double x) { int64_t b; std::memcpy(&b, &x, 8); return (int)(b & 0xffffffff); }
static inline double nmrfit_mk(int hi, int lo) {
    int64_t b = ((int64_t)hi << 32) | (uint32_t)lo; double x; std::memcpy(&x, &b, 8); return x;
}
static inline double nmrfit_rcp_seed(double q) {
    // emulate MUFU.RCP64H: only the high word of the operand is seen and only a
    // high word is produced (20 mantissa bits each way)
    double t = 1.0 / nmrfit_mk(nmrfit_hi(q), 0);
    return nmrfit_mk(nmrfit_hi(t), 0);
}
#define NMRFIT_FMA(a, b, c) std::fma((a), (b), (c))
#define NMRFIT_ABS(a) std::fabs(a)
#else
#define NMRFIT_HD __device__ __forceinline__
__device__ __forceinline__ int nmrfit_hi(double x) { return __double2hiint(x); }
__device__ __forceinline__ int nmrfit_lo(double x) { return __double2loint(x); }
__device__ __forceinline__ double nmrfit_mk(int hi, int lo) { return __hiloint2double(hi, lo); }
__device__ __forceinline__ double nmrfit_rcp_seed(double q) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(q));
    return y;
}
#define NMRFIT_FMA(a, b, c) fma((a), (b), (c))
#define NMRFIT_ABS(a) fabs(a)
#endif

namespace nmrfit {

constexpr double kPi = 3.14159265358979323846;
constexpr double kLn2 = 0.69314718055994530942;
constexpr double kSqrtLn2 = 0.83255461115769775635;          // sqrt(ln 2)
constexpr double kSqrtLn2OverPi = 0.46971863934982566689;    // sqrt(ln 2 / pi)
constexpr double kTwoOverSqrtPi = 1.12837916709551257390;    // 2 / sqrt(pi)
constexpr double kMagic = 6755399441055744.0;                // 1.5 * 2^52: round-to-nearest-int shifter
constexpr int kExpClampHi = (int)0xC085E000;                 // high word of -700.0

// The table of exp_neg<TB> in global memory (copied into shared memory by the kernels that use one); none for TB = 0
template <int TB> struct ExpTab { static NMRFIT_HD const double* src() { return nullptr; } };
template <> struct ExpTab<6> { static NMRFIT_HD const double* src() { return NMRFIT_EXP2_TAB6; } };
template <> struct ExpTab<8> { static NMRFIT_HD const double* src() { return NMRFIT_EXP2_TAB8; } };
template <> struct ExpTab<10> { static NMRFIT_HD const double* src() { return NMRFIT_EXP2_TAB10; } };

// 1/q for q >= 1 (the Lorentzian denominator 1 + t^2).  One MUFU seed with
// ~2^-20 relative error, then a cubic correction y0*(1 + e + e^2), e = 1 - q*y0:
// error ~ e^3 < 2^-57.
NMRFIT_HD double rcp_pos(double q) {
    double y0 = nmrfit_rcp_seed(q);
    double e = NMRFIT_FMA(-q, y0, 1.0);
    double g = NMRFIT_FMA(e, e, e);
    return NMRFIT_FMA(g, y0, y0);
}

template <int TB> struct ExpPoly;
template <> struct ExpPoly<0> {
    static NMRFIT_HD double eval(double r) {   // (e^r - 1)/r, degree 10
        double p = NMRFIT_EXP_T0_C10;
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T0_C9);
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T0_C8);
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T0_C7);
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T0_C6);
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T0_C5);
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T0_C4);
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T0_C3);
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T0_C2);
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T0_C1);
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T0_C0);
        return p;
    }
};
// The kernels' default table (64 entries, |r| <= ln2/128 = 5.4e-3).  Taylor coefficients of (e^r - 1)/r: the series
// is cut at r^6/720 < 3.5e-17, and 1/24 and 1/120 are TRUNCATED TO THEIR HIGH WORD (their terms are < 3.5e-11, the
// 2.4e-7 relative truncation moves the result by < 1e-17): such constants, like 1.0 and 0.5, are 32-bit immediates of
// the FP64 instructions, whereas a full 64-bit constant costs two extra instructions to materialise wherever it is
// used - and in these issue-bound kernels (DESIGN.md section 4) an integer instruction costs half an FP64 one.
template <> struct ExpPoly<6> {
    static NMRFIT_HD double eval(double r) {
        double p = 0.008333332836627960205078125;          // 1/120, high word only
        p = NMRFIT_FMA(p, r, 0.0416666567325592041015625); // 1/24, high word only
        p = NMRFIT_FMA(p, r, 0.16666666666666666);
        p = NMRFIT_FMA(p, r, 0.5);
        p = NMRFIT_FMA(p, r, 1.0);
        return p;
    }
};
template <> struct ExpPoly<8> {
    static NMRFIT_HD double eval(double r) {
        double p = NMRFIT_EXP_T8_C3;
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T8_C2);
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T8_C1);
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T8_C0);
        return p;
    }
};
template <> struct ExpPoly<10> {
    static NMRFIT_HD double eval(double r) {
        double p = NMRFIT_EXP_T10_C2;
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T10_C1);
        p = NMRFIT_FMA(p, r, NMRFIT_EXP_T10_C0);
        return p;
    }
};

// exp(x) for x <= 0 (the Gaussian) and for moderate positive x (the step ratios of
// peak_span, bounded there to < 300; nothing clamps the positive side).  Arguments
// below -700 are clamped there (exp(-700) ~ 1e-304 is zero for every purpose of a sum
// of peaks); the clamp is an unsigned min on the high word - positive doubles have a
// smaller high word and pass unchanged - i.e. integer-pipe work, not an FP64 slot.
//   n = rint(x * 2^TB / ln2);  r = x - n * ln2/2^TB  (one FMA: n*ln2/2^TB is not
//   exact, but its error n*ulp(ln2/2^TB)/2 is < 1e-16 * |x| and enters the result
//   only as a relative error of exp(x), which is itself < e^x <= 1)
//   exp(x) = 2^(n >> TB) * tab[n & (2^TB-1)] * (1 + r*P(r))
template <int TB>
NMRFIT_HD double exp_neg(double x, const double* __restrict__ tab) {
    unsigned hi = (unsigned)nmrfit_hi(x);
    hi = hi < (unsigned)kExpClampHi ? hi : (unsigned)kExpClampHi;
    x = nmrfit_mk((int)hi, nmrfit_lo(x));
    // (64/ln2 truncated to its high word for the default table: n is only the CHOICE of the table entry - the
    // reduction r = x - n*step below is exact for whatever n - and |r| grows by < 3e-7 |x| / step, 12 % at x = -700)
    constexpr double scale = TB == 6 ? 92.33245849609375 : (double)(1 << TB) / kLn2;
    constexpr double step = kLn2 / (double)(1 << TB);
    double t = NMRFIT_FMA(x, scale, kMagic);
    int n = nmrfit_lo(t);
    double nd = t - kMagic;
    double r = NMRFIT_FMA(nd, -step, x);
    double p = ExpPoly<TB>::eval(r);
    double res;
    if (TB == 0) {
        res = NMRFIT_FMA(p, r, 1.0);
    } else {
        double tj = tab[n & ((1 << TB) - 1)];
        res = NMRFIT_FMA(tj * r, p, tj);
    }
    int q = n >> TB;   // arithmetic shift: floor division for negative n
    return nmrfit_mk(nmrfit_hi(res) + (q << 20), nmrfit_lo(res));
}

// Dawson's integral F(s) = exp(-s^2) * int_0^s exp(t^2) dt, any real s (odd).
// Piecewise degree-12 polynomials on |s| < 8 (table read through the read-only
// path: lanes sit in different intervals), asymptotic form beyond: F = G(1/s^2)/(2 s) with G of degree 8 up to
// |s| = 32 and of degree 4 beyond (each to < 1e-16 relative).
NMRFIT_HD double dawson(double s, const double* __restrict__ core, const double* __restrict__ tail) {
    double as = s < 0 ? -s : s;
    double res;
    if (as < NMRFIT_DAW_SMAX) {
        int k = (int)(as * NMRFIT_DAW_INV_WIDTH);
        k = k > NMRFIT_DAW_NINT - 1 ? NMRFIT_DAW_NINT - 1 : k;
        const double* c = core + k * (NMRFIT_DAW_DEG + 1);
        double t = as - ((double)k + 0.5) * NMRFIT_DAW_WIDTH;
        double p = c[NMRFIT_DAW_DEG];
#pragma unroll
        for (int i = NMRFIT_DAW_DEG - 1; i >= 0; --i) p = NMRFIT_FMA(p, t, c[i]);
        res = p;
    } else {
        double inv = rcp_pos(as);                          // as >= 8: MUFU seed + cubic correction, no IEEE division
        double y2 = inv * inv, p;
        if (as >= NMRFIT_DAW_FAR_SMIN) {
            // far tail, a shorter polynomial: most points of a wide window are > 32 units of s from a narrow peak, and
            // neighbouring points fall on the same side of the split (generate_result is bound by these FMAs)
            const double y = y2 - NMRFIT_DAW_FAR_MID;
            p = NMRFIT_DAW_FAR[NMRFIT_DAW_FAR_DEG];
#pragma unroll
            for (int i = NMRFIT_DAW_FAR_DEG - 1; i >= 0; --i) p = NMRFIT_FMA(p, y, NMRFIT_DAW_FAR[i]);
        } else {
            const double y = y2 - NMRFIT_DAW_TAIL_MID;
            p = tail[NMRFIT_DAW_TAIL_DEG];
#pragma unroll
            for (int i = NMRFIT_DAW_TAIL_DEG - 1; i >= 0; --i) p = NMRFIT_FMA(p, y, tail[i]);
        }
        res = 0.5 * inv * p;
    }
    return s < 0 ? -res : res;
}

// ---- per-peak constants --------------------------------------------------
// voigt (reference equations.py:141-147), rewritten so the inner loop needs
// d = w - loc and d2 = d*d only:
//   L = (2/(pi W)) / (1 + d2 * (2/W)^2)            G = (2/W) sqrt(ln2/pi) exp(-d2 * (2 sqrt(ln2)/W)^2)
//   body = aL / (1 + d2*kL2) + aG * exp(d2 * nkG2)
struct PeakCoef {
    double loc;    // centre
    double kL2;    // (2/W)^2
    double aL;     // a * r * 2/(pi W)
    double nkG2;   // -(2 sqrt(ln2)/W)^2
    double aG;     // a * (1-r) * (2/W) * sqrt(ln2/pi)
};

NMRFIT_HD PeakCoef make_coef(double r, double width, double loc, double a) {
    PeakCoef c;
    double iw = 2.0 / width;
    double kg = iw * kSqrtLn2;
    c.loc = loc;
    c.kL2 = iw * iw;
    c.aL = a * r * (iw / kPi);
    c.nkG2 = -(kg * kg);
    c.aG = a * (1.0 - r) * (iw * kSqrtLn2OverPi);
    return c;
}

// ---- uniform-grid span evaluation --------------------------------------------
// On a uniformly spaced axis (w_i = w_0 + i*h: what np.linspace / a spectrometer ppm scale gives) a
// thread that owns R consecutive points evaluates a peak with far fewer instructions than one
// exponential and one reciprocal per point:
//
// Gaussian.  s_j = s_0 + j*hG (hG = h*kG), G_j = exp(-s_j^2):
//   * if no point of the span can come within |s| <= 6.5 of the centre (|s_0| > 6.5 + (R-1)|hG|), every
//     G_j < exp(-42.25) = 4.5e-19
//     of the Gaussian's height - below half an ulp of anything it is added to - and the Gaussian is
//     skipped.  With FWHM = 1.665 in s units that is ~92 % of the window for a 0.004 ppm line in a
//     0.37 ppm window;
//   * otherwise G_{j+1} = G_j * rho_j, rho_{j+1} = rho_j * c2 with rho_0 = exp(-hG*(2*s_0 + hG)),
//     c2 = exp(-2*hG^2): two exponentials per span, two multiplies per further point.  Inside the cut
//     |s_0| <= 6.5 + 4, so nothing under- or overflows.
// Lorentzian.  t_j = t_0 + j*dT (dT = h*kL), q_j = 1 + t_j^2; the reciprocals are taken four at a time
// from ONE reciprocal of q_a*q_b*q_c*q_d (Montgomery's batch inversion, with aL folded in): 13 FP64
// slots + 1 MUFU per four points instead of 16 + 4.
//
// A peak takes this path only when it is safe and accurate; the coefficient builder marks it `exact`
// otherwise, and such peaks are evaluated point by point from the STORED abscissae with one
// exponential each (peak_exact - the arithmetic of the general kernel):
//   * R*|hG| > 4: the R points of a thread span more than 4 units of s (a peak narrower than ~3 grid
//     points);
//   * kL*ulp(w) > 1e-11: treating the axis as exactly uniform moves an abscissa by up to one ulp(w)
//     against its stored value, i.e. up to kL*ulp(w) relative in a curve value - 4e-13 for a 0.004 ppm
//     line at 3.4 ppm, but it grows as the width shrinks;
//   * |t| could exceed 1e60 somewhere on the axis (the product of four q would overflow);
//   * non-finite coefficients.
constexpr double kGaussCut = 6.5;

struct SpanCoef {
    double loc, kL, kG, aL;   // centre, 2/W, 2 sqrt(ln2)/W, a r 2/(pi W)
    double aG, dT, thr, c2;   // a (1-r) (2/W) sqrt(ln2/pi), h kL, Gaussian cut for |s_0| (incl. the span), exp(-2 hG^2)
    bool exact;               // evaluate from the stored abscissae instead (peak_exact)
};

// h: axis spacing; w_ulp: 2^-52 * max|w| of the axis
NMRFIT_HD SpanCoef make_span_coef(double r, double width, double loc, double a, double h, double w_ulp, int R) {
    SpanCoef c;
    double iw = 2.0 / width;
    c.loc = loc;
    c.kL = iw;
    c.kG = iw * kSqrtLn2;
    c.aL = a * r * (iw / kPi);
    c.aG = a * (1.0 - r) * (iw * kSqrtLn2OverPi);
    c.dT = h * c.kL;
    double hG = c.dT * kSqrtLn2;
    double ah = NMRFIT_ABS(hG), ak = NMRFIT_ABS(c.kL), al = NMRFIT_ABS(loc);
    double reach = (al + w_ulp * 4503599627370496.0) * ak;     // >= |t| anywhere on the axis
    c.exact = !((double)R * ah <= 4.0 && ak * w_ulp <= 1e-11 && reach <= 1e60);   // also for NaN / inf
    c.thr = NMRFIT_FMA((double)(R - 1), ah, kGaussCut);
    c.c2 = c.exact ? 1.0 : exp_neg<0>(-2.0 * (hG * hG), nullptr);
    return c;
}

// What the span loop sees for a peak that takes the exact path: contributes exactly zero.
NMRFIT_HD SpanCoef null_span_coef() {
    SpanCoef c;
    c.loc = c.kL = c.kG = c.aL = c.aG = c.dT = 0.0;
    c.thr = -1.0;             // Gaussian never entered
    c.c2 = 1.0;
    c.exact = true;
    return c;
}

// acc[j] += aL / (1 + t_j^2) + aG * exp(-s_j^2) for the R consecutive points that start at
// distance d0 = w_first - loc from the centre (recurrence path).
template <int R, int TB>
NMRFIT_HD void peak_span(double d0, const SpanCoef& c, const double* __restrict__ tab, double (&acc)[R]) {
    static_assert(R % 4 == 0, "R must be a multiple of 4");
    const double t0 = d0 * c.kL;
    const double s0 = d0 * c.kG;
#pragma unroll
    for (int j0 = 0; j0 < R; j0 += 4) {
        const double ta = j0 == 0 ? t0 : NMRFIT_FMA((double)j0, c.dT, t0);
        const double tb = NMRFIT_FMA((double)(j0 + 1), c.dT, t0);
        const double tc = NMRFIT_FMA((double)(j0 + 2), c.dT, t0);
        const double td = NMRFIT_FMA((double)(j0 + 3), c.dT, t0);
        const double qa = NMRFIT_FMA(ta, ta, 1.0), qb = NMRFIT_FMA(tb, tb, 1.0);
        const double qc = NMRFIT_FMA(tc, tc, 1.0), qd = NMRFIT_FMA(td, td, 1.0);
        const double qab = qa * qb, qcd = qc * qd;
        const double ay = c.aL * rcp_pos(qab * qcd);
        const double yab = ay * qcd, ycd = ay * qab;      // aL/(qa qb), aL/(qc qd)
        acc[j0] = NMRFIT_FMA(yab, qb, acc[j0]);
        acc[j0 + 1] = NMRFIT_FMA(yab, qa, acc[j0 + 1]);
        acc[j0 + 2] = NMRFIT_FMA(ycd, qd, acc[j0 + 2]);
        acc[j0 + 3] = NMRFIT_FMA(ycd, qc, acc[j0 + 3]);
    }
    // Gaussian only if the span can come within the cut.  Compared on the high words (integer pipe):
    // a larger high word means a larger magnitude, equality falls on the safe side; NaN skips.
    if ((nmrfit_hi(s0) & 0x7fffffff) <= nmrfit_hi(c.thr)) {
        const double hG = c.dT * kSqrtLn2;
        double g = exp_neg<TB>(-(s0 * s0), tab);
        double rho = exp_neg<TB>(-(hG * NMRFIT_FMA(2.0, s0, hG)), tab);
#pragma unroll
        for (int j = 0; j < R; ++j) {
            acc[j] = NMRFIT_FMA(c.aG, g, acc[j]);
            if (j + 1 < R) {
                g *= rho;
                if (j + 2 < R) rho *= c.c2;
            }
        }
    }
}

// Same sum from the stored abscissae w[0..n_valid) (points past the end of the axis are extrapolated
// with h; they carry zero weight): one exponential per point, any spacing, any width.
template <int R, int TB>
NMRFIT_HD void peak_exact(const double* __restrict__ w, int n_valid, double w_first, double h, const SpanCoef& c,
                          const double* __restrict__ tab, double (&acc)[R]) {
#pragma unroll
    for (int j = 0; j < R; ++j) {
        double wj = j < n_valid ? w[j] : NMRFIT_FMA((double)j, h, w_first);
        double d = wj - c.loc;
        double t = d * c.kL, s = d * c.kG;
        double rq = rcp_pos(NMRFIT_FMA(t, t, 1.0));
        acc[j] = NMRFIT_FMA(c.aL, rq, acc[j]);
        acc[j] = NMRFIT_FMA(c.aG, exp_neg<TB>(-(s * s), tab), acc[j]);
    }
}

// ---- far field of the Lorentzians -----------------------------------------------
// Over a REGION of 2*H consecutive points (one warp's 32*R points; H = 16*R) a peak whose centre is
// far away compared with the region's half-width is a smooth function, and the sum of all such peaks
// is one polynomial.  With xi in (-1, 1) the position inside the region (xi = (i - i_c)/H), A = H*dT the
// region's half-width in t units and t_c = kL*(w_c - loc) the centre's offset,
//     aL / (1 + t^2),  t = t_c + A*xi
//   = aL * Im[ 1 / ((t_c - i) + A*xi) ]                       (1/(t - i) = (t + i)/(1 + t^2))
//   = (aL/A) * sum_n (-xi)^n Im[u^(n+1)],   u = A/(t_c - i) = A (t_c + i)/(1 + t_c^2),  |u|^2 = A^2/(1 + t_c^2)
// and v_n = Im[u^(n+1)]/A obeys v_{n+1} = 2 Re(u) v_n - |u|^2 v_{n-1}, v_{-1} = 0, v_0 = 1/(1 + t_c^2).
// A peak is FAR when |u| <= 1/16 (kFarRhoInv2 = 256) and its Gaussian cannot reach the region; the series
// is cut after kFarTerms = 12 terms, leaving < |u|^12/(1 - |u|) = 4e-15 of the Lorentzian's HEIGHT (the
// prefactor 1/A is bounded by 1/|u|), and then economised to kFarPoly = 10 coefficients (far_economise).
// Everything else is NEAR and is evaluated by peak_span.
constexpr int kFarTerms = 12;
constexpr double kFarRhoInv2 = 256.0;

// Classify one peak for a region whose centre sits Dc = w_c - loc from the peak's centre; H = half the
// region's point count.  Returns kFarNear (evaluate it with peak_span), kFarSeries (v[n] = Im[u^(n+1)]/A filled:
// the peak adds (-1)^n aL v[n] to the region's coefficient n) or kFarNothing (infinitely far: adds nothing).
enum { kFarNear = 0, kFarSeries = 1, kFarNothing = 2 };
// The part of the classification that depends on the peak and the cell LENGTH only (not on where the cell is):
// computed once per peak by the prepare pass (same expressions, same bits as far_terms evaluates on the fly).
struct FarPeak { double A, A2, A2x, reach; };                 // H dT, A^2, 256 A^2, 6.5 + H |hG|
NMRFIT_HD FarPeak make_far_peak(const SpanCoef& c, double H) {
    FarPeak f;
    f.A = H * c.dT;
    f.A2 = f.A * f.A;
    f.A2x = kFarRhoInv2 * f.A2;
    f.reach = NMRFIT_FMA(H * kSqrtLn2, NMRFIT_ABS(c.dT), kGaussCut);
    return f;
}
NMRFIT_HD int far_terms_pre(double Dc, double kL, double kG, const FarPeak& f, double (&v)[kFarTerms]) {
    const double A = f.A;
    const double tc = Dc * kL;
    const double qc = NMRFIT_FMA(tc, tc, 1.0);
    const double sc = Dc * kG;
    if (NMRFIT_ABS(sc) <= f.reach) return kFarNear;           // the Gaussian reaches the region
    if (!(f.A2x <= qc)) return kFarNear;                      // too close for the series (or NaN)
    if (!(qc <= 1e300)) return kFarNothing;                   // infinitely far: contributes nothing
    const double iq = rcp_pos(qc);
    const double two_p = 2.0 * (A * tc) * iq;                 // 2 Re(u)
    const double rho2 = f.A2 * iq;                            // |u|^2
    double vm = 0.0, vc = iq;
#pragma unroll
    for (int n = 0; n < kFarTerms; ++n) {
        v[n] = vc;
        const double vn = NMRFIT_FMA(two_p, vc, -(rho2 * vm));
        vm = vc;
        vc = vn;
    }
    return kFarSeries;
}
NMRFIT_HD int far_terms(double Dc, const SpanCoef& c, double H, double (&v)[kFarTerms]) {
    const double A = H * c.dT;
    const double tc = Dc * c.kL;
    const double qc = NMRFIT_FMA(tc, tc, 1.0);
    const double sc = Dc * c.kG;
    const double reach = NMRFIT_FMA(H * kSqrtLn2, NMRFIT_ABS(c.dT), kGaussCut);   // 6.5 + H*|hG|
    if (NMRFIT_ABS(sc) <= reach) return kFarNear;             // the Gaussian reaches the region
    if (!(kFarRhoInv2 * (A * A) <= qc)) return kFarNear;      // too close for the series (or NaN)
    if (!(qc <= 1e300)) return kFarNothing;                   // infinitely far: contributes nothing
    const double iq = rcp_pos(qc);
    const double two_p = 2.0 * (A * tc) * iq;                 // 2 Re(u)
    const double rho2 = (A * A) * iq;                         // |u|^2
    double vm = 0.0, vc = iq;
#pragma unroll
    for (int n = 0; n < kFarTerms; ++n) {
        v[n] = vc;
        const double vn = NMRFIT_FMA(two_p, vc, -(rho2 * vm));
        vm = vc;
        vc = vn;
    }
    return kFarSeries;
}

// C[n] += (-1)^n aL v[n]: one peak's series into the region's polynomial (peaks are added in index order)
NMRFIT_HD void far_add(double aL, const double (&v)[kFarTerms], double (&C)[kFarTerms]) {
#pragma unroll
    for (int n = 0; n < kFarTerms; ++n) C[n] = NMRFIT_FMA((n & 1) ? -aL : aL, v[n], C[n]);
}

// Far: adds the peak's expansion to C and returns true.  Near: returns false.
NMRFIT_HD bool far_accumulate(double Dc, const SpanCoef& c, double H, double (&C)[kFarTerms]) {
    double v[kFarTerms];
    const int kind = far_terms(Dc, c, H, v);
    if (kind == kFarNear) return false;
    if (kind == kFarSeries) far_add(c.aL, v, C);
    return true;
}

// Chebyshev economisation of the cell's polynomial.  On xi in [-1, 1]
//     x^11 = T11/1024 + (2816 x^9 - 2816 x^7 + 1232 x^5 - 220 x^3 + 11 x)/1024,
//     x^10 = T10/512  + (1280 x^8 - 1120 x^6 + 400 x^4 - 50 x^2 + 1)/512       (|T_n| <= 1),
// so dropping the T11 and T10 parts changes the polynomial by at most |C11|/1024 + |C10|/512 <= (16^-11/1024 +
// 16^-10/512) = 1.8e-15 of a far peak's height - the size of the series' own truncation error - and leaves a
// polynomial of degree 9: two FMAs fewer per point in the evaluation kernels, ten more per cell here.  The factors
// are exact binary fractions.
NMRFIT_HD void far_economise(double (&C)[kFarTerms]) {
    static_assert(kFarTerms == 12 && kFarPoly == 10, "economisation is written for 12 -> 10 coefficients");
    const double a = C[11], b = C[10];
    C[9] = NMRFIT_FMA(2.75, a, C[9]);
    C[7] = NMRFIT_FMA(-2.75, a, C[7]);
    C[5] = NMRFIT_FMA(1.203125, a, C[5]);
    C[3] = NMRFIT_FMA(-0.21484375, a, C[3]);
    C[1] = NMRFIT_FMA(0.0107421875, a, C[1]);
    C[8] = NMRFIT_FMA(2.5, b, C[8]);
    C[6] = NMRFIT_FMA(-2.1875, b, C[6]);
    C[4] = NMRFIT_FMA(0.78125, b, C[4]);
    C[2] = NMRFIT_FMA(-0.09765625, b, C[2]);
    C[0] = NMRFIT_FMA(0.001953125, b, C[0]);
}

// acc[j] = sum_n C[n] xi_j^n for the R consecutive points xi_j = xi0 + j*dxi: the accumulators START from the far
// field (the near peaks are added on top).  C: the economised polynomial (the caller may have folded a constant - the
// particle's P*yoff - into C[0]).  Split into even and odd parts, p(+-x) = E(x^2) +- x O(x^2): a thread evaluates E
// and O at its first R/2 points and gets the polynomial there AND at the mirror points -x for two more FMAs.
// far_init_half leaves p(-xi_j) in mir[j]; those are the last R/2 points (in reverse order) of the thread that holds
// the mirror image of this one's span inside the far-field cell - lane ^ (lanes per cell - 1) - which the device
// caller (uniform_eval.cuh) exchanges by shuffle: 47 FP64 instructions + 8 shuffles per thread instead of 79.
template <int R>
NMRFIT_HD void far_init_half(const double (&C)[kFarPoly], double xi0, double dxi, double (&acc)[R], double (&mir)[R / 2]) {
    static_assert(kFarPoly == 10 && R % 2 == 0, "written for a degree-9 polynomial and an even span");
#pragma unroll
    for (int j = 0; j < R / 2; ++j) {
        const double x = j == 0 ? xi0 : NMRFIT_FMA((double)j, dxi, xi0);
        const double x2 = x * x;
        double e = NMRFIT_FMA(C[8], x2, C[6]);
        double o = NMRFIT_FMA(C[9], x2, C[7]);
        e = NMRFIT_FMA(e, x2, C[4]);
        o = NMRFIT_FMA(o, x2, C[5]);
        e = NMRFIT_FMA(e, x2, C[2]);
        o = NMRFIT_FMA(o, x2, C[3]);
        e = NMRFIT_FMA(e, x2, C[0]);
        o = NMRFIT_FMA(o, x2, C[1]);
        acc[j] = NMRFIT_FMA(x, o, e);
        mir[j] = NMRFIT_FMA(-x, o, e);
    }
}

// the same on the host / for one thread alone: every point from its own abscissa, same arithmetic per point
template <int R>
NMRFIT_HD void far_init(const double (&C)[kFarPoly], double xi0, double dxi, double (&acc)[R]) {
#pragma unroll
    for (int j = 0; j < R; ++j) {
        const double x = j == 0 ? xi0 : NMRFIT_FMA((double)j, dxi, xi0);
        const double x2 = x * x;
        double e = NMRFIT_FMA(C[8], x2, C[6]);
        double o = NMRFIT_FMA(C[9], x2, C[7]);
        e = NMRFIT_FMA(e, x2, C[4]);
        o = NMRFIT_FMA(o, x2, C[5]);
        e = NMRFIT_FMA(e, x2, C[2]);
        o = NMRFIT_FMA(o, x2, C[3]);
        e = NMRFIT_FMA(e, x2, C[0]);
        o = NMRFIT_FMA(o, x2, C[1]);
        acc[j] = NMRFIT_FMA(x, o, e);
    }
}

// ---- numpy's summation order ---------------------------------------------------------------------------
// pyswarm's stop test is stepsize = np.sqrt(np.sum((g - p_min)**2)); np.sum over a contiguous float64
// vector is numpy's pairwise summation (numpy/core/src/umath/loops_utils.h.src, pairwise_sum): fewer
// than 8 elements sequentially; up to 128 elements in eight interleaved accumulators r[j] += a[i + j]
// combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) with the tail added sequentially; longer vectors split
// at n/2 rounded down to a multiple of 8.  Reproduced operation by operation, so that the comparison
// `stepsize <= minstep` sees the very value the CPU run sees.  `sq[i]` holds the rounded squares.
// LEVELS bounds the recursion: 128 << LEVELS elements (3 -> 1,024 >= 4 + 3*256 parameters).
#ifdef NMRFIT_HOST_MATH
#define NMRFIT_ADD_RN(a, b) ((a) + (b))
#else
#define NMRFIT_ADD_RN(a, b) __dadd_rn((a), (b))
#endif
template <int LEVELS>
NMRFIT_HD double numpy_pairwise_sum(const double* sq, int n) {
    if (n < 8) {
        double res = 0.0;
        for (int i = 0; i < n; ++i) res = NMRFIT_ADD_RN(res, sq[i]);
        return res;
    }
    if (LEVELS == 0 || n <= 128) {
        double r[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = sq[j];
        int i = 8;
        for (; i < n - (n % 8); i += 8) {
#pragma unroll
            for (int j = 0; j < 8; ++j) r[j] = NMRFIT_ADD_RN(r[j], sq[i + j]);
        }
        double res = NMRFIT_ADD_RN(NMRFIT_ADD_RN(NMRFIT_ADD_RN(r[0], r[1]), NMRFIT_ADD_RN(r[2], r[3])),
                                   NMRFIT_ADD_RN(NMRFIT_ADD_RN(r[4], r[5]), NMRFIT_ADD_RN(r[6], r[7])));
        for (; i < n; ++i) res = NMRFIT_ADD_RN(res, sq[i]);
        return res;
    }
    int n2 = n / 2;
    n2 -= n2 % 8;
    return NMRFIT_ADD_RN(numpy_pairwise_sum<(LEVELS > 0 ? LEVELS - 1 : 0)>(sq, n2),
                         numpy_pairwise_sum<(LEVELS > 0 ? LEVELS - 1 : 0)>(sq + n2, n - n2));
}

// Philox4x32-10 (Salmon et al., SC'11) -> two uniform doubles in [0, 1) with 53
// random bits each, built as MT19937's genrand_res53 builds them:
// (a >> 5) * 2^26 + (b >> 6), scaled by 2^-53.
struct Philox2 { double a, b; };
NMRFIT_HD void philox_round(unsigned& c0, unsigned& c1, unsigned& c2, unsigned& c3, unsigned k0, unsigned k1) {
    unsigned long long p0 = (unsigned long long)0xD2511F53u * c0;
    unsigned long long p1 = (unsigned long long)0xCD9E8D57u * c2;
    unsigned n0 = (unsigned)(p1 >> 32) ^ c1 ^ k0;
    unsigned n1 = (unsigned)p1;
    unsigned n2 = (unsigned)(p0 >> 32) ^ c3 ^ k1;
    unsigned n3 = (unsigned)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
}
NMRFIT_HD Philox2 philox_uniform2(unsigned long long seed, unsigned long long ctr_lo, unsigned long long ctr_hi) {
    unsigned c0 = (unsigned)ctr_lo, c1 = (unsigned)(ctr_lo >> 32);
    unsigned c2 = (unsigned)ctr_hi, c3 = (unsigned)(ctr_hi >> 32);
    unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        philox_round(c0, c1, c2, c3, k0, k1);
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    Philox2 o;
    o.a = ((double)(c0 >> 5) * 67108864.0 + (double)(c1 >> 6)) * (1.0 / 9007199254740992.0);
    o.b = ((double)(c2 >> 5) * 67108864.0 + (double)(c3 >> 6)) * (1.0 / 9007199254740992.0);
    return o;
}

}  // namespace nmrfit
