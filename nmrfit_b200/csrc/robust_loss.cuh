// K16 robust losses, in scipy.optimize.least_squares' convention: rho(z) of z = (res / c)^2, c = f_scale > 0 in units
// of the unweighted data (DESIGN K16).  Each loss gives, at one z,
//   rho    rho(z)
//   d1     rho'(z) > 0                  (the IRLS weight of the point is sqrt(rho'))
//   dpsi   psi'(r) = rho'(z) + 2 z rho''(z), the derivative of psi(r) = rho'(r^2/c^2) r
// Linear is least squares (rho = z): K12 keeps its own code for it (kRobust = false), so eval is never called there.
#pragma once
#include <cuda_runtime.h>
#include "../../include/nmrfit_b200.h"

namespace nmrfit {

struct LossLinear {
    static constexpr bool kRobust = false;
    static constexpr int kId = NMRFIT_LOSS_LINEAR;
    __device__ __forceinline__ static void eval(double z, double* rho, double* d1, double* dpsi) {
        *rho = z; *d1 = 1.0; *dpsi = 1.0;
    }
};

struct LossHuber {            // z for z <= 1, else 2 sqrt(z) - 1
    static constexpr bool kRobust = true;
    static constexpr int kId = NMRFIT_LOSS_HUBER;
    __device__ __forceinline__ static void eval(double z, double* rho, double* d1, double* dpsi) {
        if (z <= 1.0) {
            *rho = z; *d1 = 1.0; *dpsi = 1.0;
        } else {
            const double s = sqrt(z);
            *rho = 2.0 * s - 1.0; *d1 = 1.0 / s; *dpsi = 0.0;
        }
    }
};

struct LossSoftL1 {           // 2 (sqrt(1 + z) - 1)
    static constexpr bool kRobust = true;
    static constexpr int kId = NMRFIT_LOSS_SOFT_L1;
    __device__ __forceinline__ static void eval(double z, double* rho, double* d1, double* dpsi) {
        const double t = 1.0 + z, s = sqrt(t);
        *rho = 2.0 * (s - 1.0); *d1 = 1.0 / s; *dpsi = 1.0 / (t * s);
    }
};

struct LossCauchy {           // ln(1 + z)
    static constexpr bool kRobust = true;
    static constexpr int kId = NMRFIT_LOSS_CAUCHY;
    __device__ __forceinline__ static void eval(double z, double* rho, double* d1, double* dpsi) {
        const double t = 1.0 + z;
        *rho = log1p(z); *d1 = 1.0 / t; *dpsi = (1.0 - z) / (t * t);
    }
};

}  // namespace nmrfit
