// K14: residual autocorrelation and the lag-weighted M of the sandwich covariance (FP64, any axis)
//
// With res_i and A_i as in K12 (normal_eq_rows.cuh) and a_i = w_i^2 A_i (a row of D = 4 + 3P):
//   residual pass:  r_k = sum_{i=0}^{N-1-k} res_i res_{i+k},  k = 0..L   (the biased form: no N/(N-k) factor)
//   M pass:         M_rho = sum_i a_i^T z_i,  z_i = rho_0 a_i + sum_{k=1..L} rho_k (a_{i+k} + a_{i-k})
// with rows outside [0, N) taken as zero.  At L = 0 and rho_0 = 1, M_rho is K12's M.
//
// Mapping (a function of N, P and L only, so a spectrum's result does not depend on the batch it is in):
//   residual pass: CTA = (chunk of acf_chunk points, spectrum).  The chunk's residuals and a right halo of L more are
//     staged in shared memory; each lag is summed over `acf_segments` segments of the chunk in index order, and the
//     segments are added in order.
//   M pass: CTA = (chunk, task slice, spectrum), as K12 with one matrix.  A tile of `tp` points is staged as the rows
//     a_i of the points t0-L .. t0+tp+L-1 (L rows of halo on each side, recomputed per tile), then z of the tile's
//     points is formed by shifted sums in shared memory, and each thread adds a_i^T z_i into its 4x4 block of the
//     upper triangle.  sum a_i^T z_i is symmetric in exact arithmetic only, so the reduce writes both triangles from
//     the upper one.
//   Chunk partials of both passes are added in chunk order by a second launch.  No atomics.
#include <cuda_runtime.h>
#include <algorithm>
#include "nmrfit_internal.h"
#include "normal_eq_rows.cuh"

namespace nmrfit {

namespace {

constexpr int RB = 4;                       // register block edge
constexpr int kSmemCap = 200 * 1024 / 8;    // doubles of dynamic shared memory the M kernel opts into
constexpr int kTileTarget = 96 * 1024 / 8;  // staged rows aimed at per CTA: two CTAs per SM
constexpr int kAcfChunk = 512;
constexpr int kAcfThreads = 256;

__device__ __forceinline__ void tri_block(int q, int nb, int* bi, int* bj) {
    int i = 0;
    while (q >= nb - i) { q -= nb - i; ++i; }
    *bi = i;
    *bj = i + q;
}

__device__ __forceinline__ void load_peaks(const double* x, int P, PeakK* pk) {
    for (int k = threadIdx.x; k < P; k += blockDim.x) {
        PeakK c;
        ne_peak_constants(x, k, c);
        pk[k] = c;
    }
}

__global__ void __launch_bounds__(kAcfThreads) residual_acf_partial_kernel(const double* __restrict__ spec,
                                                                           const double* __restrict__ xs,
                                                                           LaggedPlan p, double* __restrict__ part) {
    extern __shared__ __align__(16) double smem[];
    const int b = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const int N = p.N, P = p.P, D = 4 + 3 * P, L = p.L, CH = p.acf_chunk, S = p.acf_segments;
    const double* sw = spec + (size_t)b * 4 * N;
    const double* x = xs + (size_t)b * D;
    double* res = smem;                                        // [CH + L] residuals of points c0 ..
    PeakK* pk = reinterpret_cast<PeakK*>(res + CH + L);        // [P]
    double* seg = reinterpret_cast<double*>(pk + P);           // [S][L+1] per-segment lag sums
    const double p0 = x[0], p1 = x[1], r = x[2], yoff = x[3];
    load_peaks(x, P, pk);
    __syncthreads();
    const int c0 = chunk * CH, n = min(CH, N - c0);
    const double rN = (double)N;
    for (int i = tid; i < CH + L; i += nt) {
        const int pt = c0 + i;
        if (pt >= N) { res[i] = 0.0; continue; }
        double fit = 0.0, dr = 0.0;
        for (int k = 0; k < P; ++k) {                          // peaks in index order, as K12 sums them
            double f, d;
            ne_peak_terms(pk[k], sw[pt], r, yoff, [](double, double, double) {}, &f, &d);
            fit += f;
            dr += d;
        }
        double a[4], wt, rs;
        ne_point_terms(p0, p1, pt, N, rN, sw, fit, dr, P, a, &wt, &rs);
        res[i] = rs;
    }
    __syncthreads();
    const int len = (n + S - 1) / S;
    for (int idx = tid; idx < S * (L + 1); idx += nt) {
        const int s = idx / (L + 1), k = idx - s * (L + 1);
        const int i0 = s * len, i1 = min(min(i0 + len, n), N - k - c0);     // pairs with i + k < N only
        double acc = 0.0;
        for (int i = i0; i < i1; ++i) acc = fma(res[i], res[i + k], acc);
        seg[idx] = acc;
    }
    __syncthreads();
    double* out = part + ((size_t)b * gridDim.x + chunk) * (L + 1);
    for (int k = tid; k <= L; k += nt) {
        double s = 0.0;
        for (int g = 0; g < S; ++g) s += seg[g * (L + 1) + k];
        out[k] = s;
    }
}

__global__ void residual_acf_reduce_kernel(const double* __restrict__ part, int n_chunks, int L, int B,
                                           double* __restrict__ r) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)B * (L + 1)) return;
    const int b = (int)(idx / (L + 1)), k = (int)(idx - (long long)b * (L + 1));
    const double* src = part + (size_t)b * n_chunks * (L + 1) + k;
    double s = 0.0;
    for (int c = 0; c < n_chunks; ++c) s += src[(size_t)c * (L + 1)];
    r[idx] = s;
}

__global__ void __launch_bounds__(512) lagged_m_partial_kernel(const double* __restrict__ spec,
                                                               const double* __restrict__ xs,
                                                               const double* __restrict__ rho, LaggedPlan p,
                                                               double* __restrict__ part) {
    extern __shared__ __align__(16) double smem[];
    const int b = blockIdx.z, chunk = blockIdx.x, slice = blockIdx.y;
    const int tid = threadIdx.x, nt = blockDim.x;
    const int N = p.N, P = p.P, D = 4 + 3 * P, EP = p.ep, TP = p.tp, L = p.L, R = TP + 2 * L;
    const double* sw = spec + (size_t)b * 4 * N;
    const double* x = xs + (size_t)b * D;

    double* rows = smem;                                  // [R][EP]: a rows of points t0-L .. t0+TP+L-1
    double* z = rows + R * EP;                            // [TP][EP]
    double* cdr = z + TP * EP;                            // [TP][P] per-peak d/dr terms of one group of TP rows
    PeakK* pk = reinterpret_cast<PeakK*>(cdr + TP * P);   // [P]
    double* rk = reinterpret_cast<double*>(pk + P);       // [L+1]
    double* red = smem;                                   // end of chunk: [nt][RB*RB] (aliases the rows)

    const double p0 = x[0], p1 = x[1], r = x[2], yoff = x[3];
    load_peaks(x, P, pk);
    for (int k = tid; k <= L; k += nt) rk[k] = rho[(size_t)b * (L + 1) + k];
    for (int idx = tid; idx < (R + TP) * EP; idx += nt) rows[idx] = 0.0;    // padding columns stay zero

    const int task0 = slice * p.tasks_per_slice;
    const int grp = p.ng > 1 ? tid / p.tasks : 0;
    const int task = task0 + (p.ng > 1 ? tid - grp * p.tasks : tid);
    const bool active = grp < p.ng && task < p.tasks && (p.ng > 1 || tid < p.tasks_per_slice);
    int bi = 0, bj = 0;
    if (active) tri_block(task, p.nb, &bi, &bj);
    double acc[RB][RB];
#pragma unroll
    for (int i = 0; i < RB; ++i)
#pragma unroll
        for (int j = 0; j < RB; ++j) acc[i][j] = 0.0;

    const int c0 = chunk * p.chunk, c1 = min(c0 + p.chunk, N);
    const double rN = (double)N;
    for (int t0 = c0; t0 < c1; t0 += TP) {
        // the R rows of the tile and its halo, TP at a time (the per-peak scratch holds TP rows)
        for (int g0 = 0; g0 < R; g0 += TP) {
            __syncthreads();                              // previous rows / scratch consumed (and pk, rk written)
            for (int idx = tid; idx < TP * P; idx += nt) {
                const int i = idx / P, k = idx - i * P, e = g0 + i, pt = t0 - L + e;
                if (e >= R) continue;
                double* row = rows + e * EP + 4 + 3 * k;
                if (pt < 0 || pt >= N) {
                    row[0] = row[1] = row[2] = 0.0;
                    cdr[idx] = 0.0;
                    continue;
                }
                const double wt = sw[3 * N + pt], wt2 = wt * wt;
                const PeakK c = pk[k];
                double fit;
                ne_peak_terms(c, sw[pt], r, yoff, [&](double a_gam, double a_loc, double a_area) {
                    row[0] = wt2 * a_gam; row[1] = wt2 * a_loc; row[2] = wt2 * a_area;
                }, &fit, &cdr[idx]);
            }
            __syncthreads();
            for (int i = tid; i < TP; i += nt) {
                const int e = g0 + i, pt = t0 - L + e;
                if (e >= R) continue;
                double* ra = rows + e * EP;
                if (pt < 0 || pt >= N) {
                    ra[0] = ra[1] = ra[2] = ra[3] = 0.0;
                    continue;
                }
                double dr = 0.0;
                for (int k = 0; k < P; ++k) dr += cdr[i * P + k];
                double a[4], wt, res;
                ne_point_terms(p0, p1, pt, N, rN, sw, 0.0, dr, P, a, &wt, &res);
                const double wt2 = wt * wt;
#pragma unroll
                for (int j = 0; j < 4; ++j) ra[j] = wt2 * a[j];
            }
        }
        __syncthreads();
        // z_i = rho_0 a_i + sum_k rho_k (a_{i+k} + a_{i-k}), k in order
        for (int idx = tid; idx < TP * D; idx += nt) {
            const int i = idx / D, j = idx - i * D;
            const double* c = rows + (i + L) * EP + j;
            double s = rk[0] * c[0];
            for (int k = 1; k <= L; ++k) s = fma(rk[k], c[k * EP] + c[-k * EP], s);
            z[i * EP + j] = s;
        }
        __syncthreads();
        if (active) {
            for (int i = grp; i < TP; i += p.ng) {
                const double4 av = *reinterpret_cast<const double4*>(rows + (i + L) * EP + bi * RB);
                const double4 bv = *reinterpret_cast<const double4*>(z + i * EP + bj * RB);
                const double a4[RB] = {av.x, av.y, av.z, av.w}, b4[RB] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
                for (int u = 0; u < RB; ++u)
#pragma unroll
                    for (int v = 0; v < RB; ++v) acc[u][v] = fma(a4[u], b4[v], acc[u][v]);
            }
        }
    }
    double* out = part + (((size_t)b * gridDim.x + chunk) * p.tasks) * (RB * RB);
    if (p.ng > 1) {
        __syncthreads();
        if (active)
#pragma unroll
            for (int u = 0; u < RB; ++u)
#pragma unroll
                for (int v = 0; v < RB; ++v) red[tid * RB * RB + u * RB + v] = acc[u][v];
        __syncthreads();
        for (int idx = tid; idx < p.tasks * RB * RB; idx += nt) {
            const int tk = idx / (RB * RB), e = idx - tk * (RB * RB);
            double s = 0.0;
            for (int gi = 0; gi < p.ng; ++gi) s += red[(gi * p.tasks + tk) * RB * RB + e];
            out[idx] = s;
        }
    } else if (active) {
#pragma unroll
        for (int u = 0; u < RB; ++u)
#pragma unroll
            for (int v = 0; v < RB; ++v) out[(size_t)task * RB * RB + u * RB + v] = acc[u][v];
    }
}

// fixed-order sum over chunks; one thread per (spectrum, j, k) of the D x D square, both triangles from (min, max)
__global__ void lagged_m_reduce_kernel(const double* __restrict__ part, LaggedPlan p, int B, double* __restrict__ M) {
    const int D = 4 + 3 * p.P;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)B * D * D) return;
    const int b = (int)(idx / (D * D));
    const int rem = (int)(idx - (long long)b * D * D);
    const int j0 = rem / D, k0 = rem % D;
    const int j = min(j0, k0), k = max(j0, k0);
    const int bi = j / RB, bj = k / RB;
    const int q = bi * p.nb - bi * (bi - 1) / 2 + (bj - bi);
    const double* src = part + ((size_t)b * p.n_chunks * p.tasks + q) * (RB * RB) + (j % RB) * RB + (k % RB);
    double s = 0.0;
    for (int c = 0; c < p.n_chunks; ++c) s += src[(size_t)c * p.tasks * RB * RB];
    M[idx] = s;
}

// staged doubles of the M kernel at tile tp and lag L
size_t m_stage(int tp, int L, int ep, int P) {
    return (size_t)(2 * tp + 2 * L) * ep + (size_t)tp * P + (size_t)P * (sizeof(PeakK) / sizeof(double)) + L + 1;
}

}  // namespace

LaggedPlan lagged_plan(int N, int P, int L) {
    LaggedPlan p{};
    p.N = N; p.P = P; p.L = L;
    const int D = 4 + 3 * P;
    p.nb = (D + RB - 1) / RB;
    p.ep = p.nb * RB;
    p.tasks = p.nb * (p.nb + 1) / 2;
    if (p.tasks <= 128) {                                 // few blocks: point groups share the tile
        p.ng = 256 / p.tasks;
        p.slices = 1;
        p.tasks_per_slice = p.tasks;
        p.threads = (p.ng * p.tasks + 31) / 32 * 32;
    } else {                                              // many blocks: up to 512 per CTA, the rest in further slices
        p.ng = 1;
        p.slices = (p.tasks + 511) / 512;
        p.tasks_per_slice = (p.tasks + p.slices - 1) / p.slices;
        p.threads = (p.tasks_per_slice + 31) / 32 * 32;
    }
    // the largest L whose 16-point tile fits the shared memory the kernel opts into
    const long long fixed = (long long)32 * p.ep + 16LL * P + (long long)P * (sizeof(PeakK) / sizeof(double)) + 1;
    p.max_lag = (int)std::max(0LL, ((long long)kSmemCap - fixed) / (2LL * p.ep + 1));
    int tp = 128;                                         // staged rows and halo: about 96 KB
    while (tp > 16 && m_stage(tp, L, p.ep, P) > (size_t)kTileTarget) tp /= 2;
    p.tp = tp;
    // chunk: about 2^22 Gram FMAs, between 256 points and N/128 rounded up (as K12)
    const long long target = (1LL << 22) / ((long long)D * D);
    int ch = 256;
    while ((long long)ch * 2 <= target && ch < 16384) ch *= 2;
    while ((long long)ch * 128 < N) ch *= 2;
    p.chunk = ch;
    p.n_chunks = (N + ch - 1) / ch;
    p.smem = sizeof(double) * std::max(m_stage(tp, L, p.ep, P), (size_t)p.threads * RB * RB);
    p.acf_chunk = kAcfChunk;
    p.acf_n_chunks = (N + kAcfChunk - 1) / kAcfChunk;
    p.acf_threads = kAcfThreads;
    p.acf_segments = std::max(1, kAcfThreads / (L + 1));
    p.acf_smem = sizeof(double) * ((size_t)kAcfChunk + L + (size_t)P * (sizeof(PeakK) / sizeof(double)) +
                                   (size_t)p.acf_segments * (L + 1));
    return p;
}

size_t lagged_m_scratch_doubles(const LaggedPlan& p, int B) { return (size_t)B * p.n_chunks * p.tasks * RB * RB; }

size_t residual_acf_scratch_doubles(const LaggedPlan& p, int B) {
    return (size_t)B * p.acf_n_chunks * (p.L + 1);
}

cudaError_t launch_residual_acf(const double* spec, const double* x, const LaggedPlan& p, int B, double* part,
                                double* r, cudaStream_t st) {
    residual_acf_partial_kernel<<<dim3(p.acf_n_chunks, B), p.acf_threads, p.acf_smem, st>>>(spec, x, p, part);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const long long total = (long long)B * (p.L + 1);
    residual_acf_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(part, p.acf_n_chunks, p.L, B, r);
    count_launches(2);
    return cudaGetLastError();
}

cudaError_t launch_lagged_m(const double* spec, const double* x, const double* rho, const LaggedPlan& p, int B,
                            double* part, double* M, cudaStream_t st) {
    static bool attr_set[NMRFIT_MAX_DEVICES] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_set[dev % NMRFIT_MAX_DEVICES]) {
        cudaError_t e = cudaFuncSetAttribute(lagged_m_partial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             kSmemCap * 8);
        if (e != cudaSuccess) return e;
        attr_set[dev % NMRFIT_MAX_DEVICES] = true;
    }
    lagged_m_partial_kernel<<<dim3(p.n_chunks, p.slices, B), p.threads, p.smem, st>>>(spec, x, rho, p, part);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int D = 4 + 3 * p.P;
    const long long total = (long long)B * D * D;
    lagged_m_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(part, p, B, M);
    count_launches(2);
    return cudaGetLastError();
}

}  // namespace nmrfit
