// K16 robust losses, in scipy.optimize.least_squares' convention: rho(z) of z = (res / c)^2, c = f_scale > 0 in units
// of the unweighted data (DESIGN K16).  Each loss gives, at one z,
//   rho    rho(z)
//   d1     rho'(z) > 0                  (the IRLS weight of the point is sqrt(rho'))
//   dpsi   psi'(r) = rho'(z) + 2 z rho''(z), the derivative of psi(r) = rho'(r^2/c^2) r
// Linear is least squares (rho = z): K12 keeps its own code for it (kRobust = false), so eval is never called there.
// Like nmrfit_math.cuh, the header also compiles for the host (tests/host_math_harness.cpp defines NMRFIT_HOST_MATH),
// so that the three losses can be checked against mpmath without a GPU.
#pragma once
#ifdef NMRFIT_HOST_MATH
#include <cmath>
#define NMRFIT_LOSS_HD inline
#else
#include <cuda_runtime.h>
#define NMRFIT_LOSS_HD __device__ __forceinline__
#endif
#include "../../include/nmrfit_b200.h"

namespace nmrfit {

struct LossLinear {
    static constexpr bool kRobust = false;
    static constexpr int kId = NMRFIT_LOSS_LINEAR;
    NMRFIT_LOSS_HD static void eval(double z, double* rho, double* d1, double* dpsi) {
        *rho = z; *d1 = 1.0; *dpsi = 1.0;
    }
};

struct LossHuber {            // z for z <= 1, else 2 sqrt(z) - 1
    static constexpr bool kRobust = true;
    static constexpr int kId = NMRFIT_LOSS_HUBER;
    NMRFIT_LOSS_HD static void eval(double z, double* rho, double* d1, double* dpsi) {
        if (z <= 1.0) {
            *rho = z; *d1 = 1.0; *dpsi = 1.0;
        } else {
            const double s = sqrt(z);
            *rho = 2.0 * s - 1.0; *d1 = 1.0 / s; *dpsi = 0.0;
        }
    }
};

// Each eval is within 4 ulp of the exact rho and rho', and psi' within 4 ulp of max(|psi'|, rho'), for every z in
// [0, 1e300] (tests/test_robust_loss_host.py).  That takes forms without cancellation at small z and without overflow
// at large z: 2 (sqrt(1 + z) - 1) loses all its digits to cancellation as z -> 0 (8e-5 relative at z = 1e-12, where
// c is 1e6 times the residual), and (1 + z)^2 overflows beyond z ~ 1e154 (Cauchy's psi' then came out 0).

struct LossSoftL1 {           // 2 (sqrt(1 + z) - 1) = 2 z / (sqrt(1 + z) + 1)
    static constexpr bool kRobust = true;
    static constexpr int kId = NMRFIT_LOSS_SOFT_L1;
    NMRFIT_LOSS_HD static void eval(double z, double* rho, double* d1, double* dpsi) {
        const double t = 1.0 + z, s = sqrt(t);
        *rho = 2.0 * z / (s + 1.0); *d1 = 1.0 / s; *dpsi = 1.0 / (t * s);
    }
};

struct LossCauchy {           // ln(1 + z)
    static constexpr bool kRobust = true;
    static constexpr int kId = NMRFIT_LOSS_CAUCHY;
    NMRFIT_LOSS_HD static void eval(double z, double* rho, double* d1, double* dpsi) {
        const double t = 1.0 + z, r = 1.0 / t;
        *rho = log1p(z); *d1 = r; *dpsi = (1.0 - z) * r / t;
    }
};

}  // namespace nmrfit
