// K16: moments of a robust loss at one parameter vector per spectrum (FP64, any axis)
//
// With res_i, w_i as in K12 (normal_eq_rows.cuh), c the spectrum's scale and z_i = (res_i / c)^2 (robust_loss.cuh):
//   out[b] = (s_rho = sum (w_i c sqrt(rho_i))^2,  sum (w_i res_i)^2,  sum psi_i^2,  sum psi'_i,  sum psi'_i^2)
// with psi_i = rho'(z_i) res_i and psi'_i = rho'(z_i) + 2 z_i rho''(z_i).  For LossLinear: (w res)^2 twice, psi = res,
// psi' = 1.  These give the refined fit's weighted RMSE and the scale factor of Huber's sandwich covariance (DESIGN K16).
//
// Mapping (a function of N only, as K14's residual pass): CTA = (chunk of kChunk points, spectrum); thread t adds the
// points c0 + t, c0 + t + nt, ... in that order, the threads' sums are added in thread order, and a second launch adds
// the chunks in chunk order.  No atomics.
#include <cuda_runtime.h>
#include "nmrfit_internal.h"
#include "normal_eq_rows.cuh"
#include "robust_loss.cuh"

namespace nmrfit {

namespace {

constexpr int kChunk = 512;
constexpr int kThreads = 256;
constexpr int kMoments = 5;

template <typename Loss>
__global__ void __launch_bounds__(kThreads) loss_moments_partial_kernel(const double* __restrict__ spec,
                                                                        const double* __restrict__ xs,
                                                                        const double* __restrict__ fscale, int N,
                                                                        int P, double* __restrict__ part) {
    extern __shared__ __align__(16) double smem[];
    const int b = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x, nt = blockDim.x, D = 4 + 3 * P;
    const double* sw = spec + (size_t)b * 4 * N;
    const double* x = xs + (size_t)b * D;
    PeakK* pk = reinterpret_cast<PeakK*>(smem);                        // [P]
    double* red = reinterpret_cast<double*>(pk + P);                   // [nt][kMoments]
    const double p0 = x[0], p1 = x[1], r = x[2], yoff = x[3];
    for (int k = tid; k < P; k += nt) {
        PeakK c;
        ne_peak_constants(x, k, c);
        pk[k] = c;
    }
    __syncthreads();
    const double c = Loss::kRobust ? fscale[b] : 1.0;
    const int c0 = chunk * kChunk, c1 = min(c0 + kChunk, N);
    const double rN = (double)N;
    double m[kMoments] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int pt = c0 + tid; pt < c1; pt += nt) {
        double wt, res;
        ne_residual(pk, P, p0, p1, r, yoff, pt, N, rN, sw, &wt, &res);
        const double wr = wt * res;
        double q = wr, psi = res, dpsi = 1.0;
        if constexpr (Loss::kRobust) {
            const double zr = res / c;
            double rho, d1;
            Loss::eval(zr * zr, &rho, &d1, &dpsi);
            q = wt * c * sqrt(rho);
            psi = d1 * res;
        }
        m[0] = fma(q, q, m[0]);
        m[1] = fma(wr, wr, m[1]);
        m[2] = fma(psi, psi, m[2]);
        m[3] += dpsi;
        m[4] = fma(dpsi, dpsi, m[4]);
    }
#pragma unroll
    for (int k = 0; k < kMoments; ++k) red[tid * kMoments + k] = m[k];
    __syncthreads();
    if (tid < kMoments) {
        double s = 0.0;
        for (int t = 0; t < nt; ++t) s += red[t * kMoments + tid];
        part[((size_t)b * gridDim.x + chunk) * kMoments + tid] = s;
    }
}

__global__ void loss_moments_reduce_kernel(const double* __restrict__ part, int n_chunks, int B,
                                           double* __restrict__ out) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * kMoments) return;
    const int b = idx / kMoments, k = idx - b * kMoments;
    const double* src = part + (size_t)b * n_chunks * kMoments + k;
    double s = 0.0;
    for (int ch = 0; ch < n_chunks; ++ch) s += src[(size_t)ch * kMoments];
    out[idx] = s;
}

template <typename Loss>
cudaError_t launch_moments(const double* spec, const double* x, const double* fscale, int B, int N, int P,
                           double* part, double* out, cudaStream_t st) {
    const int n_chunks = (N + kChunk - 1) / kChunk;
    const size_t smem = sizeof(PeakK) * P + sizeof(double) * kThreads * kMoments;
    loss_moments_partial_kernel<Loss><<<dim3(n_chunks, B), kThreads, smem, st>>>(spec, x, fscale, N, P, part);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    loss_moments_reduce_kernel<<<(B * kMoments + 255) / 256, 256, 0, st>>>(part, n_chunks, B, out);
    count_launches(2);
    return cudaGetLastError();
}

}  // namespace

size_t loss_moments_scratch_doubles(int B, int N) { return (size_t)B * ((N + kChunk - 1) / kChunk) * kMoments; }

cudaError_t launch_loss_moments(const double* spec, const double* x, int loss, const double* fscale, int B, int N,
                                int P, double* part, double* out, cudaStream_t st) {
    switch (loss) {
    case NMRFIT_LOSS_HUBER: return launch_moments<LossHuber>(spec, x, fscale, B, N, P, part, out, st);
    case NMRFIT_LOSS_SOFT_L1: return launch_moments<LossSoftL1>(spec, x, fscale, B, N, P, part, out, st);
    case NMRFIT_LOSS_CAUCHY: return launch_moments<LossCauchy>(spec, x, fscale, B, N, P, part, out, st);
    default: return launch_moments<LossLinear>(spec, x, fscale, B, N, P, part, out, st);
    }
}

}  // namespace nmrfit
