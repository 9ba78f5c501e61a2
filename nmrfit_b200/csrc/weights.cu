// K8: residual weights for a batch of spectra, on the device.
//
// Reference: FitUtility._compute_weights (utils.py:191-224) + equations.laplace1d (equations.py:215-238), run
// once per fit on the host.  For a batch of spectra (BASELINE config 3) it is the only per-spectrum host work
// left, so it moves next to the data:
//   1. per peak, the index window [argmin|w - b0|, argmin|w - b1|] (swapped if reversed; utils.py:206-211),
//      np.argmin's first-occurrence rule;
//   2. weights = 1, then each peak's window is set to its value (tallest/|height|)**expon in peak order - later
//      peaks overwrite earlier ones (utils.py:220-221).  The P values per spectrum are computed by the caller
//      on the host (P calls of pow; keeps them bit-identical to numpy's);
//   3. n Jacobi sweeps x[1:-1] = (1-omega) x[1:-1] + (omega*0.5) (x[2:] + x[:-2]) with pinned ends, every
//      operation rounded separately exactly as numpy evaluates the expression.
// One CTA per spectrum; the sweeps ping-pong between the context's weights plane and a scratch plane.
// Integer/compare work plus 4 flop per point per sweep: bound by L2/HBM traffic of 16 B per point per sweep.
#include <cuda_runtime.h>
#include <math_constants.h>
#include "nmrfit_internal.h"

namespace nmrfit {

constexpr int kWThreads = 1024;

__global__ void __launch_bounds__(kWThreads)
weights_kernel(double* __restrict__ spec, double* __restrict__ scratch, const double* __restrict__ bounds,
               const double* __restrict__ values, int N, int n_windows, int sweeps, double one_minus_omega,
               double half_omega) {
    extern __shared__ int win[];                           // [n_windows][2] lo, hi; then values as doubles
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = kWThreads / 32;
    double* sval = reinterpret_cast<double*>(win + 2 * ((n_windows + 1) & ~1));
    const double* w = spec + (size_t)b * 4 * N;
    double* wt = spec + (size_t)b * 4 * N + 3 * (size_t)N;
    double* sc = scratch + (size_t)b * N;

    // 1. one warp per (peak, bound): first index of the smallest |w - bound|
    for (int t = warp; t < 2 * n_windows; t += NW) {
        const double target = bounds[(size_t)b * 2 * n_windows + t];
        double bf = CUDART_INF;
        int bi = 0x7fffffff;
        for (int i = lane; i < N; i += 32) {
            const double d = fabs(w[i] - target);
            if (d < bf) { bf = d; bi = i; }                // strict: the earlier index of this lane stays
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double of = __shfl_xor_sync(0xffffffffu, bf, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (of < bf || (of == bf && oi < bi)) { bf = of; bi = oi; }
        }
        if (lane == 0) win[t] = bi == 0x7fffffff ? 0 : bi;  // all-NaN: np.argmin returns 0
    }
    for (int k = tid; k < n_windows; k += kWThreads) sval[k] = values[(size_t)b * n_windows + k];
    __syncthreads();
    for (int k = tid; k < n_windows; k += kWThreads) {     // utils.py:208-211: order the pair
        const int a = win[2 * k], c = win[2 * k + 1];
        win[2 * k] = min(a, c);
        win[2 * k + 1] = max(a, c);
    }
    __syncthreads();

    // 2. fill: the LAST peak whose window holds the point wins
    for (int i = tid; i < N; i += kWThreads) {
        double x = 1.0;
        for (int k = 0; k < n_windows; ++k)
            if (i >= win[2 * k] && i <= win[2 * k + 1]) x = sval[k];
        wt[i] = x;
    }
    __syncthreads();

    // 3. Jacobi sweeps, ends pinned
    double* src = wt;
    double* dst = sc;
    for (int s = 0; s < sweeps; ++s) {
        for (int i = tid; i < N; i += kWThreads) {
            double x = src[i];
            if (i > 0 && i < N - 1)
                x = __dadd_rn(__dmul_rn(one_minus_omega, x), __dmul_rn(half_omega, __dadd_rn(src[i + 1], src[i - 1])));
            dst[i] = x;
        }
        __syncthreads();
        double* t = src; src = dst; dst = t;
    }
    if (src != wt) {
        for (int i = tid; i < N; i += kWThreads) wt[i] = src[i];
    }
}

cudaError_t launch_weights(double* spec, double* scratch, const double* bounds_dev, const double* values_dev, int B,
                           int N, int n_windows, int sweeps, double omega, cudaStream_t st) {
    const size_t smem = sizeof(int) * 2 * ((n_windows + 1) & ~1) + sizeof(double) * n_windows;
    if (smem > 48 * 1024) {                                // up to 4,096 windows (64 KB): beyond the default limit
        cudaError_t e = opt_in_smem<weights_kernel>(80 * 1024);
        if (e != cudaSuccess) return e;
    }
    // numpy evaluates (1. - omega) * x[1:-1] + omega * 0.5 * (x[2:] + x[:-2]) with the scalars folded first
    weights_kernel<<<B, kWThreads, smem, st>>>(spec, scratch, bounds_dev, values_dev, N, n_windows, sweeps, 1.0 - omega,
                                               omega * 0.5);
    count_launches(1);
    return cudaGetLastError();
}

}  // namespace nmrfit
