// Host build of nmrfit_b200/csrc/nmrfit_math.cuh and robust_loss.cuh for accuracy tests without a GPU.
// Compiled by tests/test_host_math.py and tests/test_robust_loss_host.py with g++ into a shared object;
// the product never links or loads it.
#define NMRFIT_HOST_MATH 1
#define __device__
#define __host__
#define __constant__
#define __forceinline__ inline
#include <vector>
#include "../nmrfit_b200/csrc/nmrfit_math.cuh"
#include "../nmrfit_b200/csrc/robust_loss.cuh"

// Loss::eval of one loss (NMRFIT_LOSS_*) at z[0..n): rho, rho' and psi' = rho' + 2 z rho''
template <typename Loss>
static void loss_eval(const double* z, int n, double* rho, double* d1, double* dpsi) {
    for (int i = 0; i < n; ++i) Loss::eval(z[i], rho + i, d1 + i, dpsi + i);
}

// Sum of peaks over a uniform grid w_i = w[0] + i*h, evaluated span by span exactly as
// objective_uniform_kernel does it: anchors at the true w of every R-th point.
template <int R, int TB>
static void spans(const double* w, int n, double h, const double* x, int P, const double* tab, double* vfit) {
    double big = std::fabs(w[0]) > std::fabs(w[n - 1]) ? std::fabs(w[0]) : std::fabs(w[n - 1]);
    const double w_ulp = 2.220446049250313e-16 * big;
    for (int i0 = 0; i0 < n; i0 += R) {
        double acc[R];
        for (int j = 0; j < R; ++j) acc[j] = (double)P * x[3];
        for (int k = 0; k < P; ++k) {
            nmrfit::SpanCoef c = nmrfit::make_span_coef(x[2], x[4 + 3 * k], x[5 + 3 * k], x[6 + 3 * k], h, w_ulp, R);
            if (!c.exact) nmrfit::peak_span<R, TB>(w[i0] - c.loc, c, tab, acc);
            else nmrfit::peak_exact<R, TB>(w + i0, n - i0, w[i0], h, c, tab, acc);
        }
        for (int j = 0; j < R && i0 + j < n; ++j) vfit[i0 + j] = acc[j];
    }
}

// The same sum as `spans`, with the far-field split of objective_uniform_kernel: regions of 32*R points,
// near peaks by peak_span / peak_exact, far peaks through one polynomial per region.
template <int R, int TB>
static void regions(const double* w, int n, double h, const double* x, int P, const double* tab, double* vfit,
                    int* n_near_total) {
    double big = std::fabs(w[0]) > std::fabs(w[n - 1]) ? std::fabs(w[0]) : std::fabs(w[n - 1]);
    const double w_ulp = 2.220446049250313e-16 * big;
    const int RG = 32 * R;
    const double H = 16.0 * R;
    int near_total = 0;
    for (int r0 = 0; r0 < n; r0 += RG) {
        const double wc = std::fma(0.5 * (RG - 1), h, w[r0]);
        double C[nmrfit::kFarTerms] = {0};
        std::vector<int> near;
        std::vector<nmrfit::SpanCoef> cs(P);
        for (int k = 0; k < P; ++k) {
            cs[k] = nmrfit::make_span_coef(x[2], x[4 + 3 * k], x[5 + 3 * k], x[6 + 3 * k], h, w_ulp, R);
            if (cs[k].exact || !nmrfit::far_accumulate(wc - cs[k].loc, cs[k], H, C)) near.push_back(k);
        }
        near_total += (int)near.size();
        nmrfit::far_economise(C);                              // 12 series terms -> 10 stored coefficients
        double Ce[nmrfit::kFarPoly];
        for (int n2 = 0; n2 < nmrfit::kFarPoly; ++n2) Ce[n2] = C[n2];
        for (int lane = 0; lane < 32; ++lane) {
            const int i0 = r0 + lane * R;
            if (i0 >= n) break;
            double acc[R];
            const double xi0 = ((double)(lane * R) - 0.5 * (RG - 1)) / H;
            nmrfit::far_init<R>(Ce, xi0, 1.0 / H, acc);       // the accumulators start from the far field
            for (int k : near) {
                if (!cs[k].exact) nmrfit::peak_span<R, TB>(w[i0] - cs[k].loc, cs[k], tab, acc);
                else nmrfit::peak_exact<R, TB>(w + i0, n - i0, w[i0], h, cs[k], tab, acc);
            }
            for (int j = 0; j < R && i0 + j < n; ++j) vfit[i0 + j] = acc[j] + (double)P * x[3];
        }
    }
    *n_near_total = near_total;
}

extern "C" {

int h_region_fit(const double* w, int n, double h, const double* x, int P, int R, double* vfit) {
    int near = 0;
    if (R == 4) regions<4, 6>(w, n, h, x, P, NMRFIT_EXP2_TAB6, vfit, &near);
    else if (R == 8) regions<8, 6>(w, n, h, x, P, NMRFIT_EXP2_TAB6, vfit, &near);
    else regions<16, 6>(w, n, h, x, P, NMRFIT_EXP2_TAB6, vfit, &near);
    return near;
}

// the 12-term far-field polynomial at x[0..n) by Horner (`full`) and after far_economise, by the even/odd form the
// kernels evaluate (`econ`: far_init on one point at a time)
void h_far_poly(const double* C12, const double* x, int n, double* full, double* econ) {
    double C[nmrfit::kFarTerms], Ce[nmrfit::kFarPoly];
    for (int k = 0; k < nmrfit::kFarTerms; ++k) C[k] = C12[k];
    for (int i = 0; i < n; ++i) {
        double p = C[nmrfit::kFarTerms - 1];
        for (int k = nmrfit::kFarTerms - 2; k >= 0; --k) p = std::fma(p, x[i], C[k]);
        full[i] = p;
    }
    nmrfit::far_economise(C);
    for (int k = 0; k < nmrfit::kFarPoly; ++k) Ce[k] = C[k];
    for (int i = 0; i + 1 < n; i += 2) {
        double acc[2];
        nmrfit::far_init<2>(Ce, x[i], x[i + 1] - x[i], acc);
        econ[i] = acc[0];
        econ[i + 1] = acc[1];
    }
}

void h_exp_neg(int tb, const double* x, int n, double* out) {
    for (int i = 0; i < n; ++i) {
        switch (tb) {
            case 0: out[i] = nmrfit::exp_neg<0>(x[i], nullptr); break;
            case 6: out[i] = nmrfit::exp_neg<6>(x[i], NMRFIT_EXP2_TAB6); break;
            case 8: out[i] = nmrfit::exp_neg<8>(x[i], NMRFIT_EXP2_TAB8); break;
            default: out[i] = nmrfit::exp_neg<10>(x[i], NMRFIT_EXP2_TAB10); break;
        }
    }
}

void h_rcp_pos(const double* q, int n, double* out) {
    for (int i = 0; i < n; ++i) out[i] = nmrfit::rcp_pos(q[i]);
}

void h_dawson(const double* s, int n, double* out) {
    for (int i = 0; i < n; ++i) out[i] = nmrfit::dawson(s[i], NMRFIT_DAW_TAB, NMRFIT_DAW_TAIL);
}

// body of one peak at the points w (same association as the kernels use)
void h_voigt_body(const double* w, int n, double r, double width, double loc, double a, int tb, double* out) {
    nmrfit::PeakCoef c = nmrfit::make_coef(r, width, loc, a);
    for (int i = 0; i < n; ++i) {
        double d = w[i] - c.loc, d2 = d * d;
        double q = NMRFIT_FMA(d2, c.kL2, 1.0);
        double acc = c.aL * nmrfit::rcp_pos(q);
        double e = tb == 0 ? nmrfit::exp_neg<0>(d2 * c.nkG2, nullptr) : nmrfit::exp_neg<6>(d2 * c.nkG2, NMRFIT_EXP2_TAB6);
        out[i] = NMRFIT_FMA(c.aG, e, acc);
    }
}

void h_span_fit(const double* w, int n, double h, const double* x, int P, int R, int tb, double* vfit) {
    if (tb == 6) {
        if (R == 4) spans<4, 6>(w, n, h, x, P, NMRFIT_EXP2_TAB6, vfit);
        else if (R == 8) spans<8, 6>(w, n, h, x, P, NMRFIT_EXP2_TAB6, vfit);
        else spans<16, 6>(w, n, h, x, P, NMRFIT_EXP2_TAB6, vfit);
    } else {
        if (R == 4) spans<4, 10>(w, n, h, x, P, NMRFIT_EXP2_TAB10, vfit);
        else if (R == 8) spans<8, 10>(w, n, h, x, P, NMRFIT_EXP2_TAB10, vfit);
        else spans<16, 10>(w, n, h, x, P, NMRFIT_EXP2_TAB10, vfit);
    }
}

void h_loss(int loss, const double* z, int n, double* rho, double* d1, double* dpsi) {
    switch (loss) {
        case NMRFIT_LOSS_HUBER: loss_eval<nmrfit::LossHuber>(z, n, rho, d1, dpsi); break;
        case NMRFIT_LOSS_SOFT_L1: loss_eval<nmrfit::LossSoftL1>(z, n, rho, d1, dpsi); break;
        case NMRFIT_LOSS_CAUCHY: loss_eval<nmrfit::LossCauchy>(z, n, rho, d1, dpsi); break;
        default: loss_eval<nmrfit::LossLinear>(z, n, rho, d1, dpsi); break;
    }
}

double h_numpy_sum(const double* sq, int n) { return nmrfit::numpy_pairwise_sum<3>(sq, n); }

void h_philox(unsigned long long seed, unsigned long long lo, unsigned long long hi, double* out2) {
    nmrfit::Philox2 p = nmrfit::philox_uniform2(seed, lo, hi);
    out2[0] = p.a; out2[1] = p.b;
}

}
