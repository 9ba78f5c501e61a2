// K12: normal equations of the objective at one parameter vector per spectrum (FP64, any axis)
//
// With res_i = Vdata_i(p0, p1) - Vfit_i(x) and A_i = d res_i / dx (a row of D = 4 + 3P), accumulate over the N points
//   H = sum w_i^2 A_i^T A_i,   M = sum w_i^4 A_i^T A_i,   g = sum w_i^2 res_i A_i,   ssr = (sum w_i^2 res_i^2, sum res_i^2).
// Both are Gram matrices of E = D + 1 columns: H_ext of the rows [w A, w res] (H, g and ssr_w in its last column) and
// M_ext of the rows [w^2 A, res] (M, and sum res^2 in its corner; its last column repeats g and is dropped).
//
// Mapping (a function of N and D only, so a spectrum's result does not depend on the batch it is in):
//   CTA = (chunk of `chunk` points, task slice, spectrum).  A tile of `tp` points is staged in shared memory as the
//   scaled rows of both matrices; each thread owns one RB x RB block of the upper triangle of one matrix in registers
//   (a symmetric rank-tp update per tile: RB^2 DFMA per 2*RB shared loads).  When the blocks are fewer than the
//   threads, `ng` point groups split the tile's points and are added in group order at the end of the chunk.
//   Chunk partials [B][n_chunks][tasks][RB*RB] are added in chunk order by the second launch.  No atomics.
//
// K16, robust losses (robust_loss.cuh, DESIGN K16): the same pass with every H_ext row scaled by sqrt(rho'(z_i)),
// z_i = (res_i / c)^2, so that H holds H_rho = sum w^2 rho' A^T A and g holds g_rho = sum w^2 rho' res A, and the last
// column of the M_ext row set to q_i = w_i c sqrt(rho(z_i)), whose corner is the cost s_rho = sum w^2 c^2 rho.  The
// plan is K12's.  Out block: H_rho | M (K12's) | g_rho | ssr = (s_rho, sum w^2 rho' res^2): the two corners swap
// places, so the step kernel finds the cost where it finds s.  Loss = LossLinear is K12 (same SASS).
#include <cuda_runtime.h>
#include <algorithm>
#include "nmrfit_internal.h"
#include "normal_eq_rows.cuh"
#include "robust_loss.cuh"

namespace nmrfit {

namespace {

constexpr int RB = 4;                  // register block edge

// upper-triangle block q of an nb x nb block grid -> (row block, column block), row-major over bi <= bj
__device__ __forceinline__ void tri_block(int q, int nb, int* bi, int* bj) {
    int i = 0;
    while (q >= nb - i) { q -= nb - i; ++i; }
    *bi = i;
    *bj = i + q;
}

// fscale [B]: the loss's scale c of each spectrum (not read by LossLinear)
template <typename Loss>
__global__ void __launch_bounds__(512) normal_eq_partial_kernel(const double* __restrict__ spec,
                                                                const double* __restrict__ xs, NormalEqPlan p,
                                                                double* __restrict__ part,
                                                                const double* __restrict__ fscale) {
    extern __shared__ __align__(16) double smem[];
    const int b = blockIdx.z, chunk = blockIdx.x, slice = blockIdx.y;
    const int tid = threadIdx.x, nt = blockDim.x;
    const int N = p.N, P = p.P, D = 4 + 3 * P, EP = p.ep, TP = p.tp;
    const double* sw = spec + (size_t)b * 4 * N;
    const double* x = xs + (size_t)b * D;

    double* rows = smem;                                  // [2][TP][EP]: H_ext rows, then M_ext rows
    double* cfit = rows + 2 * TP * EP;                    // [TP][P]  per-peak model values
    double* cdr = cfit + TP * P;                          // [TP][P]  per-peak d/dr terms
    PeakK* pk = reinterpret_cast<PeakK*>(cdr + TP * P);   // [P]
    double* red = smem;                                   // end of chunk: [nt][RB*RB] (aliases the rows)

    const double p0 = x[0], p1 = x[1], r = x[2], yoff = x[3];
    for (int k = tid; k < P; k += nt) {
        PeakK c;
        ne_peak_constants(x, k, c);
        pk[k] = c;
    }
    for (int idx = tid; idx < 2 * TP * EP; idx += nt) rows[idx] = 0.0;    // padding columns stay zero

    // this thread's block of the Gram matrices
    const int task0 = slice * p.tasks_per_slice;
    const int grp = p.ng > 1 ? tid / p.tasks : 0;
    const int task = task0 + (p.ng > 1 ? tid - grp * p.tasks : tid);
    const bool active = grp < p.ng && task < p.tasks && (p.ng > 1 || tid < p.tasks_per_slice);
    int mat = 0, bi = 0, bj = 0;
    if (active) {
        mat = task / p.tri;
        tri_block(task - mat * p.tri, p.nb, &bi, &bj);
    }
    double acc[RB][RB];
#pragma unroll
    for (int i = 0; i < RB; ++i)
#pragma unroll
        for (int j = 0; j < RB; ++j) acc[i][j] = 0.0;

    const int c0 = chunk * p.chunk, c1 = min(c0 + p.chunk, N);
    const double rN = (double)N;
    for (int t0 = c0; t0 < c1; t0 += TP) {
        __syncthreads();                                  // previous tile's rows are consumed (and pk is written)
        // (point, peak) pairs: the three peak columns of A, the model value and the d/dr term
        for (int idx = tid; idx < TP * P; idx += nt) {
            const int i = idx / P, k = idx - i * P, pt = t0 + i;
            double* row = rows + i * EP + 4 + 3 * k;
            double* rowm = row + TP * EP;
            if (pt >= c1) {
                row[0] = row[1] = row[2] = rowm[0] = rowm[1] = rowm[2] = 0.0;
                cfit[idx] = cdr[idx] = 0.0;
                continue;
            }
            const double wt = sw[3 * N + pt], wt2 = wt * wt;
            const PeakK c = pk[k];
            ne_peak_terms(c, sw[pt], r, yoff, [&](double a_gam, double a_loc, double a_area) {
                row[0] = wt * a_gam; row[1] = wt * a_loc; row[2] = wt * a_area;
                rowm[0] = wt2 * a_gam; rowm[1] = wt2 * a_loc; rowm[2] = wt2 * a_area;
            }, &cfit[idx], &cdr[idx]);
        }
        __syncthreads();
        // per point: phase, residual, the four global columns; peaks summed in index order
        for (int i = tid; i < TP; i += nt) {
            const int pt = t0 + i;
            double* rh = rows + i * EP;
            double* rm = rh + TP * EP;
            if (pt >= c1) {
                rh[0] = rh[1] = rh[2] = rh[3] = rh[D] = rm[0] = rm[1] = rm[2] = rm[3] = rm[D] = 0.0;
                continue;
            }
            double fit = 0.0, dr = 0.0;
            for (int k = 0; k < P; ++k) {
                fit += cfit[i * P + k];
                dr += cdr[i * P + k];
            }
            double a[4], wt, res;
            ne_point_terms(p0, p1, pt, N, rN, sw, fit, dr, P, a, &wt, &res);
            const double wt2 = wt * wt;
            if constexpr (Loss::kRobust) {
                // the IRLS weight is known only now: the peak columns written above are scaled here too
                const double c = fscale[b], zr = res / c;
                double rho, d1, dpsi;
                Loss::eval(zr * zr, &rho, &d1, &dpsi);
                const double sr = sqrt(d1);
                for (int j = 4; j < D; ++j) rh[j] *= sr;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    rh[j] = (wt * a[j]) * sr;
                    rm[j] = wt2 * a[j];
                }
                rh[D] = (wt * res) * sr;
                rm[D] = wt * c * sqrt(rho);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    rh[j] = wt * a[j];
                    rm[j] = wt2 * a[j];
                }
                rh[D] = wt * res;
                rm[D] = res;
            }
        }
        __syncthreads();
        if (active) {
            const double* base = rows + mat * TP * EP;
            for (int i = grp; i < TP; i += p.ng) {
                const double* ri = base + i * EP;
                const double4 av = *reinterpret_cast<const double4*>(ri + bi * RB);
                const double4 bv = *reinterpret_cast<const double4*>(ri + bj * RB);
                const double a4[RB] = {av.x, av.y, av.z, av.w}, b4[RB] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
                for (int u = 0; u < RB; ++u)
#pragma unroll
                    for (int v = 0; v < RB; ++v) acc[u][v] = fma(a4[u], b4[v], acc[u][v]);
            }
        }
    }
    // point groups added in group order, then one block per task to the chunk's partials
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

// fixed-order sum over chunks; one thread per (spectrum, matrix, j, k) of the E x E square, both triangles
// (kRobust: the corner of M_ext, the cost, goes to ssr[0] and that of H_ext to ssr[1])
template <bool kRobust>
__global__ void normal_eq_reduce_kernel(const double* __restrict__ part, NormalEqPlan p, int n_chunks, int B,
                                        double* __restrict__ out) {
    const int D = 4 + 3 * p.P, E = D + 1;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)B * 2 * E * E) return;
    const int b = (int)(idx / (2 * E * E));
    const int rem = (int)(idx - (long long)b * 2 * E * E);
    const int mat = rem / (E * E), j0 = (rem / E) % E, k0 = rem % E;
    if (mat == 1 && (j0 == D) != (k0 == D)) return;      // M_ext's last column repeats g
    const int j = min(j0, k0), k = max(j0, k0);
    const int bi = j / RB, bj = k / RB;
    const int q = bi * p.nb - bi * (bi - 1) / 2 + (bj - bi);
    const int task = mat * p.tri + q, e = (j % RB) * RB + (k % RB);
    const double* src = part + ((size_t)b * n_chunks * p.tasks + task) * (RB * RB) + e;
    double s = 0.0;
    for (int c = 0; c < n_chunks; ++c) s += src[(size_t)c * p.tasks * RB * RB];
    // out per spectrum block: H [D][D], M [D][D], g [D], ssr [2]
    const size_t DD = (size_t)D * D;
    double* o = out + (size_t)b * (2 * DD + D + 2);
    if (j0 < D && k0 < D) o[mat * DD + (size_t)j0 * D + k0] = s;
    else if (mat == 0 && j0 < D) o[2 * DD + j0] = s;     // (j0, D) of H_ext: g
    else if (j0 == D && k0 == D) o[2 * DD + D + (kRobust ? 1 - mat : mat)] = s;
}

}  // namespace

NormalEqPlan normal_eq_plan(int N, int P) {
    NormalEqPlan p{};
    p.N = N; p.P = P;
    const int D = 4 + 3 * P, E = D + 1;
    p.nb = (E + RB - 1) / RB;
    p.ep = p.nb * RB;
    p.tri = p.nb * (p.nb + 1) / 2;
    p.tasks = 2 * p.tri;
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
    int tp = 128;                                         // staged rows of both matrices: about 48 KB
    while (tp > 16 && 2 * tp * p.ep > 6144) tp /= 2;
    p.tp = tp;
    // chunk: about 2^22 Gram FMAs per matrix, between 256 points and N/128 rounded up
    const long long target = (1LL << 22) / ((long long)E * E);
    int ch = 256;
    while ((long long)ch * 2 <= target && ch < 16384) ch *= 2;
    while ((long long)ch * 128 < N) ch *= 2;
    p.chunk = ch;
    p.n_chunks = (N + ch - 1) / ch;
    const size_t stage = (size_t)2 * tp * p.ep + (size_t)2 * tp * P + (size_t)P * (sizeof(PeakK) / sizeof(double));
    p.smem = sizeof(double) * std::max(stage, (size_t)p.threads * RB * RB);
    return p;
}

size_t normal_eq_scratch_doubles(const NormalEqPlan& p, int B) {
    return (size_t)B * p.n_chunks * p.tasks * RB * RB;
}

namespace {

template <typename Loss>
cudaError_t launch_pass(const double* spec, const double* x, const double* fscale, const NormalEqPlan& p, int B,
                        double* part, double* out, cudaStream_t st) {
    static bool attr_set[NMRFIT_MAX_DEVICES] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_set[dev % NMRFIT_MAX_DEVICES]) {
        cudaError_t e = cudaFuncSetAttribute(normal_eq_partial_kernel<Loss>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        attr_set[dev % NMRFIT_MAX_DEVICES] = true;
    }
    dim3 grid(p.n_chunks, p.slices, B);
    normal_eq_partial_kernel<Loss><<<grid, p.threads, p.smem, st>>>(spec, x, p, part, fscale);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int E = 5 + 3 * p.P;
    const long long total = (long long)B * 2 * E * E;
    normal_eq_reduce_kernel<Loss::kRobust><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(part, p, p.n_chunks, B,
                                                                                            out);
    count_launches(2);
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_normal_eq(const double* spec, const double* x, const NormalEqPlan& p, int B, double* part,
                             double* out, cudaStream_t st) {
    return launch_pass<LossLinear>(spec, x, nullptr, p, B, part, out, st);
}

cudaError_t launch_normal_eq_loss(const double* spec, const double* x, int loss, const double* fscale,
                                  const NormalEqPlan& p, int B, double* part, double* out, cudaStream_t st) {
    switch (loss) {
    case NMRFIT_LOSS_HUBER: return launch_pass<LossHuber>(spec, x, fscale, p, B, part, out, st);
    case NMRFIT_LOSS_SOFT_L1: return launch_pass<LossSoftL1>(spec, x, fscale, p, B, part, out, st);
    case NMRFIT_LOSS_CAUCHY: return launch_pass<LossCauchy>(spec, x, fscale, p, B, part, out, st);
    default: return launch_normal_eq(spec, x, p, B, part, out, st);
    }
}

}  // namespace nmrfit
