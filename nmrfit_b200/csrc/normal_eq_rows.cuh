// Row arithmetic of the linearised residual, shared by the normal-equations pass (K12, normal_eq.cu) and the lagged
// passes (K14, lagged.cu), so that every pass sees the same residual and the same Jacobian row at a point.
//
// With res_i = Vdata_i(p0, p1) - Vfit_i(x) and A_i = d res_i / dx (D = 4 + 3P columns):
//   per (point, peak): the peak's three columns of A, its model value and its d/dr term   (ne_peak_terms)
//   per point:         the phase, the residual and the four global columns                 (ne_point_terms)
// The model value and the d/dr term are summed over the peaks in index order by the caller.
// The statement order here (columns handed to the caller before the model value is formed, the weight loaded after the
// phase) is the order K12 had before it was factored out: its SASS is byte-identical to that version.
#pragma once
#include <cuda_runtime.h>

namespace nmrfit {

constexpr double kNeSqrtLn2 = 0.83255461115769775635;
constexpr double kNeSqrtLn2OverPi = 0.46971863934982566;   // sqrt(ln 2 / pi)
constexpr double kNeInvPi = 0.31830988618379067154;

struct PeakK { double loc, gam, area, kL, kG, cL, cG, igam; };

// constants of peak k of x = [p0, p1, r, yoff, (width, loc, area) x P]
__device__ __forceinline__ void ne_peak_constants(const double* x, int k, PeakK& c) {
    c.gam = x[4 + 3 * k]; c.loc = x[5 + 3 * k]; c.area = x[6 + 3 * k];
    c.igam = 1.0 / c.gam;
    c.kL = 2.0 * c.igam;
    c.kG = 2.0 * kNeSqrtLn2 * c.igam;
    c.cL = c.kL * kNeInvPi;
    c.cG = c.kL * kNeSqrtLn2OverPi;
}

// one (point, peak) pair at axis value wp: columns(d res / d width, d res / d loc, d res / d area), then the peak's
// model value area * mix + yoff and its d/dr term area * (L - G)
template <typename Columns>
__device__ __forceinline__ void ne_peak_terms(const PeakK& c, double wp, double r, double yoff, Columns&& columns,
                                              double* fit, double* dr) {
    const double d = wp - c.loc;
    const double t = d * c.kL, s = d * c.kG;
    const double q = fma(t, t, 1.0);
    const double iq = 1.0 / q;
    const double L = c.cL * iq;
    const double G = c.cG * exp(-(s * s));
    const double mix = fma(r, L, (1.0 - r) * G);
    const double dl_loc = L * (2.0 * t) * iq * c.kL, dg_loc = G * (2.0 * s) * c.kG;
    const double dl_gam = L * c.igam * (fma(t, t, -1.0) * iq), dg_gam = G * c.igam * fma(2.0 * s, s, -1.0);
    columns(-c.area * fma(r, dl_gam, (1.0 - r) * dg_gam), -c.area * fma(r, dl_loc, (1.0 - r) * dg_loc), -mix);
    *fit = fma(c.area, mix, yoff);
    *dr = c.area * (L - G);
}

// point pt of the N in sw = [w | u | v | weights] with the model summed over the peaks (fit) and its d/dr (dr): the
// global columns d res / d(p0, p1, r, yoff) in a[4], the point's weight and its residual
__device__ __forceinline__ void ne_point_terms(double p0, double p1, int pt, int N, double rN, const double* sw,
                                               double fit, double dr, int P, double a[4], double* wt, double* res) {
    double sn, cs;
    sincos(p0 + (p1 * (double)pt) / rN, &sn, &cs);
    const double u = sw[N + pt], v = sw[2 * N + pt];
    const double vd = fma(u, cs, -(v * sn)), id = fma(u, sn, v * cs);
    a[0] = -id;
    a[1] = -id * ((double)pt / rN);
    a[2] = -dr;
    a[3] = -(double)P;
    *wt = sw[3 * N + pt];
    *res = vd - fit;
}

}  // namespace nmrfit
